"""SoundStream VQ-VAE -- host-side mirror of the reference ``models/vq_brain.py``.

Same class names, constructor kwargs, ``forward`` signatures, return conventions and state-dict
keys as the reference (models/vq_brain.py:22-243), so this module drops into
``notebooks_trainer/vq_brain_trainer.ipynb`` and ``utils/train_utils.py:138``.  What changes
underneath:

* the quantiser is ``frankenstein_b200.vector_quantize.VectorQuantize`` (tcgen05 search + fused
  epilogue kernels) instead of the third-party ``vector_quantize_pytorch`` module;
* ``custom_l1_loss`` is one fused masked-sum kernel (no ``nonzero`` host sync, no dynamic shape);
* ``calculate_perp`` is computed from the code histogram (no ``[N, K]`` one-hot).

* the causal conv / transposed-conv stacks (SURVEY.md section 8f row N1) run channels-last on the library's tcgen05
  GEMMs as implicit GEMMs (``conv.py``: ``[B, T, C]`` activations, im2col rows are overlapping views of the padded
  signal) whenever every layer's channel counts are multiples of 64; other widths, and ``FK_CONV=cudnn``, use cuDNN's
  NHWC kernels on a 4-D view (no permute copies either way).

* ``SoundStream.stream`` (no reference counterpart) tokenizes a recording online, 4 bins at a time, on the same implicit
  GEMMs with a per-layer history of input rows (``TokenizerStream``).
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, conv, gemm, ops
from ._lib import DTYPE_CODE, FkError, check, counters, lib, on_tensor_device, ptr, require_cuda, require_device, stream
from .vector_quantize import VectorQuantize, finish, prepare_codebook, prepare_input, search


# "own" (default): the conv stacks run channels-last on the library's tcgen05 GEMMs (conv.py: im2col rows are overlapping
# views of the padded signal); "cudnn": the same stacks as 1 x k conv2d on cuDNN's NHWC kernels (A/B comparison only).
CONV_IMPL = os.environ.get("FK_CONV", "own")
_CL3D = [False]      # set by _ChannelsFirstStack while its layers run on [B, T, C] activations


def _own_conv_ok(m) -> bool:
    return (m.padding_mode == "zeros" and conv.conv_supported(m.in_channels, m.out_channels, m.kernel_size[0], m.stride[0],
                                                             m.dilation[0], m.groups))


class CausalConv1d(nn.Conv1d):
    """models/vq_brain.py:22-28 -- left padding of dilation * (k - 1)."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.causal_padding = self.dilation[0] * (self.kernel_size[0] - 1)

    def forward(self, x):
        if _CL3D[0] and x.dim() == 3:                       # [B, T, C]: implicit GEMM on tcgen05 (conv.py)
            return conv.causal_conv1d_cl(x, self.weight, self.bias, self.stride[0])
        if x.dim() == 4:
            # channels-last path ([B, C, 1, T] with NHWC strides, see _ChannelsFirstStack): the same convolution as a
            # 1 x k conv2d, so that cuDNN runs its NHWC kernels without a layout conversion before and after
            return F.conv2d(F.pad(x, [self.causal_padding, 0]), self.weight.unsqueeze(2), self.bias,
                            stride=(1, self.stride[0]), dilation=(1, self.dilation[0]), groups=self.groups)
        return self._conv_forward(F.pad(x, [self.causal_padding, 0]), self.weight, self.bias)


class CausalConvTranspose1d(nn.ConvTranspose1d):
    """models/vq_brain.py:31-45 -- transposed conv with the trailing k - s samples trimmed."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.causal_padding = (self.dilation[0] * (self.kernel_size[0] - 1) + self.output_padding[0] + 1
                               - self.stride[0])

    def forward(self, x, output_size=None):
        if self.padding_mode != 'zeros':
            raise ValueError('Only `zeros` padding mode is supported for ConvTranspose1d')
        if _CL3D[0] and x.dim() == 3:
            return conv.causal_conv_transpose1d_cl(x, self.weight, self.bias)
        if x.dim() == 4:                                    # channels-last path (see CausalConv1d)
            y = F.conv_transpose2d(x, self.weight.unsqueeze(2), self.bias, stride=(1, self.stride[0]),
                                   padding=(0, self.padding[0]), output_padding=(0, self.output_padding[0]),
                                   groups=self.groups, dilation=(1, self.dilation[0]))
            return y[..., :-self.causal_padding]
        output_padding = self._output_padding(x, output_size, self.stride, self.padding, self.kernel_size,
                                              self.dilation)
        y = F.conv_transpose1d(x, self.weight, self.bias, self.stride, self.padding, output_padding, self.groups,
                               self.dilation)
        return y[..., :-self.causal_padding]


class _PointwiseConv1d(nn.Conv1d):
    """nn.Conv1d (same parameters / state-dict keys) that also takes the channels-last 4-D layout."""

    def forward(self, x):
        if _CL3D[0] and x.dim() == 3:                       # 1 x 1 convolution = the plain projection of the channel axis
            return gemm.linear(x, self.weight.squeeze(2), self.bias)
        if x.dim() == 4:
            return F.conv2d(x, self.weight.unsqueeze(2), self.bias, stride=(1, self.stride[0]),
                            padding=(0, self.padding[0]), dilation=(1, self.dilation[0]), groups=self.groups)
        return super().forward(x)


def _interleave_elu(mods):
    """[m0, ELU, m1, ELU, ..., mN] -- the Sequential indexing the reference checkpoints expect."""
    out = []
    for i, m in enumerate(mods):
        if i:
            out.append(nn.ELU())
        out.append(m)
    return nn.Sequential(*out)


class ResidualUnit(nn.Module):
    """x + Conv1x1(ELU(CausalConv3(x)))  (models/vq_brain.py:48-63)."""

    def __init__(self, in_channels, out_channels, dilation):
        super().__init__()
        self.dilation = dilation
        self.layers = _interleave_elu([
            CausalConv1d(in_channels, out_channels, kernel_size=3, dilation=dilation),
            _PointwiseConv1d(out_channels, in_channels, kernel_size=1),
        ])

    def forward(self, x):
        return x + self.layers(x)


def _residual_stack(ch, n=3):
    return [ResidualUnit(ch, ch, dilation=1) for _ in range(n)]


class EncoderBlock(nn.Module):
    """3 residual units then a strided causal conv (k = 2*stride)  (models/vq_brain.py:66-90)."""

    def __init__(self, in_channels, out_channels, stride):
        super().__init__()
        self.layers = _interleave_elu(_residual_stack(in_channels) + [
            CausalConv1d(in_channels, out_channels, kernel_size=2 * stride, stride=stride)])

    def forward(self, x):
        return self.layers(x)


class DecoderBlock(nn.Module):
    """strided causal transposed conv then 3 residual units  (models/vq_brain.py:93-117)."""

    def __init__(self, in_channels, out_channels, stride):
        super().__init__()
        self.layers = _interleave_elu([
            CausalConvTranspose1d(in_channels, out_channels, kernel_size=2 * stride, stride=stride)]
            + _residual_stack(out_channels))

    def forward(self, x):
        return self.layers(x)


class _ChannelsFirstStack(nn.Module):
    """[B, T, C] in and out.  The reference permutes to [B, C, T] (vq_brain.py:135-137, 156-158) and cuDNN then converts
    to NHWC and back around every convolution.  Here [B, T, C] is viewed, without a copy, as the channels-last 4-D tensor
    [B, C, 1, T] (its NHWC strides are exactly those of a contiguous [B, T, C]), every layer is the equivalent 1 x k
    conv2d, and the result is viewed back: no permute copies and no layout-conversion kernels."""

    def _own_ok(self) -> bool:
        if getattr(self, "_own_checked", None) is None:
            ok = True
            for m in self.modules():
                if isinstance(m, CausalConv1d):
                    ok = ok and _own_conv_ok(m)
                elif isinstance(m, CausalConvTranspose1d):
                    ok = ok and (m.kernel_size[0] == 4 and m.stride[0] == 2 and m.dilation[0] == 1 and m.groups == 1
                                 and m.output_padding[0] == 0 and m.in_channels % 32 == 0 and m.out_channels % 32 == 0)
                elif isinstance(m, _PointwiseConv1d):
                    ok = ok and (m.kernel_size[0] == 1 and m.stride[0] == 1 and m.groups == 1
                                 and gemm.linear_supported(m.in_channels, m.out_channels))
            self._own_checked = ok
        return self._own_checked

    def forward(self, x):
        if x.is_cuda and x.dim() == 3 and CONV_IMPL == "own" and self._own_ok():
            # activations stay [B, T, C] bf16: every convolution is an implicit GEMM over overlapping-row views (conv.py),
            # no permutes, no im2col copies, no cuDNN
            _CL3D[0] = True
            try:
                return self.layers(x)
            finally:
                _CL3D[0] = False
        if x.is_cuda and x.dim() == 3 and x.is_contiguous():
            y = self.layers(x.transpose(1, 2).unsqueeze(2))          # [B, C, 1, T], channels_last strides
            return y.squeeze(2).transpose(1, 2)
        return self.layers(x.transpose(1, 2)).transpose(1, 2)


class Encoder(_ChannelsFirstStack):
    """models/vq_brain.py:120-138: conv k5 -> 2 x EncoderBlock(stride 2) -> conv k3; T/4 tokens of width D."""

    def __init__(self, C, D, n_electrodes):
        super().__init__()
        self.layers = _interleave_elu([
            CausalConv1d(n_electrodes, C, kernel_size=5),
            EncoderBlock(C, C, stride=2),
            EncoderBlock(C, C, stride=2),
            CausalConv1d(C, D, kernel_size=3),
        ])


class Decoder(_ChannelsFirstStack):
    """models/vq_brain.py:141-159: mirror of the encoder."""

    def __init__(self, C, D, n_channels_out):
        super().__init__()
        self.layers = _interleave_elu([
            CausalConv1d(D, C, kernel_size=3),
            DecoderBlock(C, C, stride=2),
            DecoderBlock(C, C, stride=2),
            CausalConv1d(C, n_channels_out, kernel_size=5),
        ])


class _MaskedL1(torch.autograd.Function):
    """custom_l1_loss (models/vq_brain.py:220-227) as one fused forward and one fused backward kernel."""

    @staticmethod
    @on_tensor_device
    def forward(ctx, pred, gt):
        require_cuda(pred, gt)
        require_device()
        ctx.pred_dtype = pred.dtype
        if pred.dtype not in (torch.float32, torch.bfloat16):
            pred = pred.float()
        B, T, C = pred.shape
        p = pred.contiguous()
        g = gt.contiguous().float()
        R = B * T
        nb = lib().fk_masked_l1_partials(R)
        dev = pred.device
        row_valid = torch.empty(R, device=dev, dtype=torch.uint8)
        ps = torch.empty(nb, device=dev, dtype=torch.float32)
        pc = torch.empty(nb, device=dev, dtype=torch.float32)
        loss = torch.empty(1, device=dev, dtype=torch.float32)
        denom = torch.empty(1, device=dev, dtype=torch.float32)
        check(lib().fk_masked_l1_forward(ptr(p), DTYPE_CODE[p.dtype], ptr(g), R, C, ptr(row_valid), ptr(ps), ptr(pc),
                                         counters(_lib.CTR_MASKED_L1), ptr(loss), ptr(denom), stream()), "fk_masked_l1_forward")
        ctx.save_for_backward(p, g, row_valid, denom)
        return loss.view(())

    @staticmethod
    @on_tensor_device
    def backward(ctx, g_loss):
        p, g, row_valid, denom = ctx.saved_tensors
        B, T, C = p.shape
        grad = torch.empty_like(p)
        gl = g_loss.reshape(1).contiguous().float()
        check(lib().fk_masked_l1_backward(ptr(p), DTYPE_CODE[p.dtype], ptr(g), ptr(row_valid), ptr(gl), ptr(denom), B * T,
                                          C, ptr(grad), stream()), "fk_masked_l1_backward")
        return grad.to(ctx.pred_dtype), None


@on_tensor_device
def perplexity(indices: torch.Tensor, codebook_size: int) -> torch.Tensor:
    """calculate_perp (models/vq_brain.py:238-243) from the code histogram."""
    require_cuda(indices)
    require_device()
    ind = indices.reshape(-1).contiguous()
    bins = torch.empty(codebook_size, device=ind.device, dtype=torch.float32)
    out = torch.empty(1, device=ind.device, dtype=torch.float32)
    check(lib().fk_vq_perplexity(ptr(ind), ind.numel(), codebook_size, ptr(bins), ptr(out), stream()), "fk_vq_perplexity")
    return out.view(())


class SoundStream(nn.Module):
    """models/vq_brain.py:162-243.  forward(x[B,T,n_electrodes]) -> (rec_loss + commit_loss [1], o [B,T,n_electrodes])."""

    def __init__(self, C, D, codebook_size, n_electrodes, use_cosine_sim=True):
        super().__init__()
        self.codebook_size = codebook_size
        self.encoder = Encoder(C=C, D=D, n_electrodes=n_electrodes)
        self.quantizer = VectorQuantize(
            dim=D,
            codebook_size=codebook_size,
            commitment_weight=0.25,
            channel_last=True,
            kmeans_init=True,
            threshold_ema_dead_code=2,
            use_cosine_sim=use_cosine_sim,
        )
        self.decoder = Decoder(C=C, D=D, n_channels_out=n_electrodes)
        self.compute_perplexity = False     # the reference computes it and discards the value (vq_brain.py:212)
        self.last_perplexity = None

    def forward(self, x, targets=None, date_info=None):
        e = self.encoder(x)
        quantized, indices, commit_loss = self.quantizer(e)
        if quantized.dtype != e.dtype and not torch.is_autocast_enabled():
            quantized = quantized.to(e.dtype)      # module cast to bf16/fp16 without autocast
        o = self.decoder(quantized)
        if self.compute_perplexity:
            self.last_perplexity = self.calculate_perp(indices)
        rec_loss = self.custom_l1_loss(o, x)
        total_loss = rec_loss + commit_loss
        return total_loss, o

    def custom_l1_loss(self, pred, gt):
        return _MaskedL1.apply(pred, gt)

    def get_quantize_vectors(self, x):
        e = self.encoder(x)
        quantized, indices, commit_loss = self.quantizer(e)
        return indices, quantized

    def calculate_perp(self, indices):
        return perplexity(indices, self.codebook_size)

    def stream(self, batch_size: int, reconstruct: bool = False) -> "TokenizerStream":
        """Online tokenization: feed a recording 4 bins at a time (or any multiple of 4) with `TokenizerStream.step(x)` and
        get the codes of the new bins only, at a cost that does not grow with the length of the stream.

        Every layer of the stacks is causal -- CausalConv1d pads on the left only and CausalConvTranspose1d trims its
        trailing samples (models/vq_brain.py:22-45) -- so the output for bin t never changes once bin t has arrived, and
        each convolution needs only its last k - 1 input rows (1 for the transposed convolution) from earlier steps.  The
        encoder's receptive field is 44 bins: token t reads bins 4t - 40 ... 4t + 3.

        The stream converts every weight and the codebook once, here: it tokenizes with the model as it is now.  After
        training or loading new weights, create a new stream."""
        return TokenizerStream(self, batch_size, reconstruct)


# ------------------------------------------------------------------------------------------------
# streaming inference (SoundStream.stream)
# ------------------------------------------------------------------------------------------------
class _PlanEntry:
    """One convolution of a flattened stack: its input rows are act(x + r), x = the previous entry's output, r = the input
    rows of entry `res` (a ResidualUnit's `x + layers(x)`) or none; `hist` = taps - 1 input rows carried between steps."""
    __slots__ = ("conv", "taps", "hist", "stride", "transposed", "elu", "res")

    def __init__(self, conv_, taps, stride, transposed, elu, res):
        self.conv, self.taps, self.hist, self.stride = conv_, taps, taps - 1, stride
        self.transposed, self.elu, self.res = transposed, elu, res


def _stream_plan(stack: nn.Module):
    """Flatten an Encoder / Decoder into its convolutions in order ([_PlanEntry]), checking every module against the
    structure the stream reproduces: FkError for anything else (other module types or subclasses, other activations, an
    ELU that does not feed a convolution, dilated / grouped / padded convolutions, a ResidualUnit that changes the rate or
    the width)."""
    if type(stack) not in (Encoder, Decoder):
        raise FkError(f"SoundStream.stream: cannot stream a {type(stack).__name__}")
    plan = []
    pending = {"elu": False, "res": None}

    def conv_entry(m, taps, stride, transposed):
        if m.dilation[0] != 1 or m.groups != 1 or m.padding[0] != 0 or m.padding_mode != "zeros":
            raise FkError(f"SoundStream.stream: {type(m).__name__} with dilation, groups or padding cannot stream")
        plan.append(_PlanEntry(m, taps, stride, transposed, pending["elu"], pending["res"]))
        pending["elu"], pending["res"] = False, None

    def walk(seq):
        if type(seq) is not nn.Sequential:
            raise FkError(f"SoundStream.stream: expected an nn.Sequential of layers, got {type(seq).__name__}")
        for m in seq:
            t = type(m)
            if t is nn.ELU:
                if m.alpha != 1.0 or pending["elu"] or not plan:
                    raise FkError("SoundStream.stream: an ELU (alpha 1) must follow a layer and feed a convolution")
                pending["elu"] = True
            elif t is CausalConv1d:
                k, s = m.kernel_size[0], m.stride[0]
                if not (s == 1 or (s == 2 and k == 4)):
                    raise FkError(f"SoundStream.stream: CausalConv1d k = {k}, stride {s} cannot stream")
                conv_entry(m, k, s, False)
            elif t is CausalConvTranspose1d:
                if m.kernel_size[0] != 4 or m.stride[0] != 2 or m.output_padding[0] != 0:
                    raise FkError("SoundStream.stream: CausalConvTranspose1d must be k = 4, stride 2")
                conv_entry(m, 2, 1, True)          # two taps of [x[v-1] | x[v]], output rows [y[2v] | y[2v+1]]
            elif t is _PointwiseConv1d:
                if m.kernel_size[0] != 1 or m.stride[0] != 1:
                    raise FkError("SoundStream.stream: a 1 x 1 convolution must have stride 1")
                conv_entry(m, 1, 1, False)
            elif t is ResidualUnit:
                start = len(plan)               # the unit's input = the input rows of its first convolution
                walk(m.layers)
                inner = plan[start:]
                if (not inner or pending["elu"] or pending["res"] is not None
                        or any(e.stride != 1 or e.transposed for e in inner)
                        or inner[0].conv.in_channels != inner[-1].conv.out_channels):
                    raise FkError("SoundStream.stream: a ResidualUnit must keep the rate and width and end in a convolution")
                pending["res"] = start
            elif t in (EncoderBlock, DecoderBlock):
                walk(m.layers)
            else:
                raise FkError(f"SoundStream.stream: cannot stream a {t.__name__}")

    walk(stack.layers)
    if not plan or pending["elu"] or pending["res"] is not None:
        raise FkError("SoundStream.stream: the stack must end in a convolution")
    return plan


class _StreamLayer:
    """A plan entry with its weights converted once (bf16 GEMM layout, fp32 bias) and its two history buffers."""

    def __init__(self, e: _PlanEntry, batch_size: int, device):
        m = e.conv
        self.e = e
        if e.transposed:
            self.w2, self.bias = conv._w_transpose_pairs(m.weight, m.bias)
        else:
            self.w2 = conv._w_taps_major(m.weight)
            self.bias = None if m.bias is None else m.bias.detach().float().clone()
        self.hist = (torch.zeros(2, batch_size, e.hist, m.in_channels, device=device, dtype=torch.bfloat16)
                     if e.hist else None)


class TokenizerStream:
    """Streaming state of a `SoundStream` (from `SoundStream.stream`): per convolution of the encoder (and, with
    `reconstruct`, of the decoder) the last taps - 1 input rows in bf16, two buffers each -- a step reads one and writes
    the other, and the roles swap only once the whole step has been enqueued, so a rejected step leaves the state as it
    was.  Weights and codebook are a snapshot taken at creation.

    With per-row `counts` each row advances by its own number of bins.  The counts reach the device once per step, as a
    table of the count at each rate of the stacks (bins, half, quarter = tokens); each convolution reads the row of its
    input rate, so a row's rows past its count never reach a GEMM and its histories advance by its own rows only."""

    def __init__(self, model: SoundStream, batch_size: int, reconstruct: bool = False):
        if batch_size < 1:
            raise FkError("TokenizerStream: batch_size must be positive")
        stacks = [model.encoder] + ([model.decoder] if reconstruct else [])
        plans = [_stream_plan(s) for s in stacks]
        dev = next(model.parameters()).device
        if dev.type != "cuda":
            raise FkError("frankenstein_b200 modules run on a B200 only (no CPU fallback)")
        if not all(s._own_ok() for s in stacks):
            raise FkError("TokenizerStream: a convolution width is outside the library's implicit GEMMs (cuDNN-only widths "
                          "cannot stream)")
        vq = model.quantizer
        if not vq._is_initted():
            raise FkError("TokenizerStream: the codebook is not initialised (k-means on a stream chunk is meaningless); "
                          "train the model or load a checkpoint first")
        self.batch_size, self.reconstruct, self.device = batch_size, bool(reconstruct), dev
        self.n_electrodes = model.encoder.layers[0].in_channels
        self.use_cosine = vq.use_cosine_sim
        with torch.cuda.device(dev):
            self._layers = [[_StreamLayer(e, batch_size, dev) for e in p] for p in plans]
            self._embed = vq.codebook.detach().float().clone().contiguous()
            self._cb, self._c2pad = prepare_codebook(self._embed, self.use_cosine)
        self._cur = 0
        self._lengths = [0] * batch_size

    @property
    def lengths(self) -> list:
        """bins consumed so far, per row (each row is a recording of its own; see `reset`)."""
        return list(self._lengths)

    @property
    def length(self) -> int:
        """bins consumed so far, while every row is at the same position."""
        return ops.stream_length(self._lengths, "TokenizerStream.length")

    def reset(self, rows=None) -> None:
        """Start a new recording in every row (rows None) or only in the given row indices: their histories become the
        causal zero padding again, and the other rows carry on untouched.  FkError, changing nothing, for an index outside
        the batch or a duplicate."""
        if rows is None:
            for layers in self._layers:
                for L in layers:
                    if L.hist is not None:
                        L.hist.zero_()
            self._lengths = [0] * self.batch_size
            return
        idx = ops.stream_rows(rows, self.batch_size, "TokenizerStream.reset")
        if not idx:
            return
        dev_idx = torch.tensor(idx, dtype=torch.long).to(self.device)
        for layers in self._layers:
            for L in layers:
                if L.hist is not None:
                    L.hist.index_fill_(1, dev_idx, 0)          # both buffers of the rows
        for r in idx:
            self._lengths[r] = 0

    def _run(self, layers, x, cnt=None, level=0):
        """cnt: None or device int32 [3, B], row k the rows' counts at 1 / 2^k of the bin rate; level: the rate of x."""
        inputs = []
        cur = self._cur
        for L in layers:
            e = L.e
            r = None if e.res is None else inputs[e.res]
            h_in, h_out = (None, None) if L.hist is None else (L.hist[cur], L.hist[cur ^ 1])
            y, rows = conv.causal_conv1d_step(x, r, e.elu, h_in, h_out, L.w2, L.bias, e.taps, e.stride,
                                              None if cnt is None else cnt[level])
            if e.transposed:
                y = y.reshape(y.shape[0], 2 * y.shape[1], y.shape[2] // 2)
                level -= 1
            elif e.stride == 2:
                level += 1
            inputs.append(rows)
            x = y
        return x

    @torch.no_grad()
    def step(self, x: torch.Tensor, counts=None):
        """x [B, 4n, n_electrodes] (fp32 or bf16, n >= 1) -> (indices [B, n] int64, quantized [B, n, D] fp32), plus, with
        `reconstruct`, the decoder output o [B, 4n, n_electrodes] (bf16) of the new bins.  The quantizer runs with eval
        semantics whatever the model's mode (no k-means, no EMA update).

        counts: optional host sequence of B ints, the bins of x that are new data for each row (0 ... 4n, multiples of 4).
        Row b advances by counts[b] bins; the rest of its bins are ignored whatever they hold (NaN included).  Past a row's
        count its indices are -1, its quantized vectors zero and its decoder bins zero; a count of 0 leaves the row's
        histories bit for bit as they were.  None, or every count 4n, is the plain step.

        Raises FkError, leaving the state as it was, on a bin count that is not a positive multiple of 4, a batch or channel
        count that does not match the stream, bad counts (number, range, multiples of 4), a CPU tensor or a dtype other
        than fp32 / bf16."""
        B, E = self.batch_size, self.n_electrodes
        if not isinstance(x, torch.Tensor) or x.dim() != 3 or x.shape[0] != B or x.shape[2] != E:
            raise FkError(f"TokenizerStream.step: expected [{B}, 4n, {E}], got "
                          f"{tuple(x.shape) if isinstance(x, torch.Tensor) else type(x).__name__}")
        T = x.shape[1]
        if T < 4 or T % 4 != 0:
            raise FkError(f"TokenizerStream.step: {T} bins is not a positive multiple of 4")
        if not x.is_cuda:
            raise FkError("frankenstein_b200 modules run on a B200 only (no CPU fallback)")
        if x.device != self.device:
            raise FkError(f"TokenizerStream.step: the stream lives on {self.device}, x on {x.device}")
        if x.dtype not in (torch.float32, torch.bfloat16):
            raise FkError(f"TokenizerStream.step: x must be fp32 or bf16, got {x.dtype}")
        if counts is not None:
            counts = ops.stream_counts(counts, B, T, 4, "TokenizerStream.step")
            if all(c == T for c in counts):
                counts = None                          # every row takes the whole step: the plain step
        if x.stride(2) != 1 or x.stride(0) % 8 or x.stride(1) % 8 or x.data_ptr() % 16:
            x = x.contiguous()
        n = T // 4
        with torch.cuda.device(self.device):
            cnt = None
            if counts is not None:
                # one host-to-device copy: the counts at the bin, half and token rates of the stacks
                cnt = torch.tensor([counts, [c // 2 for c in counts], [c // 4 for c in counts]],
                                   dtype=torch.int32).to(self.device)
            e = self._run(self._layers[0], x.detach(), cnt, 0)
            D = e.shape[2]
            xn, xb, _ = prepare_input(e.reshape(B * n, D).contiguous(), self.use_cosine)
            cand_val, cand_idx = search(xb, self._cb, self._c2pad, self._embed.shape[0], self.use_cosine)
            indices, quantized, _ = finish(xn, self._embed, cand_val, cand_idx, self.use_cosine, False, 0.0)
            out = (indices.view(B, n), quantized.view(B, n, D))
            if cnt is not None:
                past = torch.arange(n, device=self.device)[None] >= cnt[2][:, None]       # token slots past the counts
                out[0].masked_fill_(past, -1)
                out[1].masked_fill_(past[..., None], 0)
            if self.reconstruct:
                o = self._run(self._layers[1], out[1], cnt, 2)
                if cnt is not None:
                    o.masked_fill_((torch.arange(T, device=self.device)[None] >= cnt[0][:, None])[..., None], 0)
                out = out + (o,)
        self._cur ^= 1
        self._lengths = [m + a for m, a in zip(self._lengths, [T] * B if counts is None else counts)]
        return out
