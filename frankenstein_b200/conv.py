"""SoundStream's causal convolutions as channels-last implicit GEMMs on the library's tcgen05 kernels (SURVEY section 8f,
row N1; reference: models/vq_brain.py:22-45 CausalConv1d / CausalConvTranspose1d and the stacks built from them, :48-159).

Activations stay ``[B, T, C]`` (time-major, channels contiguous) in bf16 through a whole stack -- the layout the reference
permutes away from (vq_brain.py:135-137, 156-158).  In that layout the im2col row of output step t of a dilation-1 convolution,
``x_pad[b, t*s : t*s + k, :]``, is a CONTIGUOUS run of k*C_in elements of the left-padded signal, so the whole im2col matrix is a
strided VIEW with overlapping rows (row stride s*C_in) and the convolution is one NT GEMM ``A_view [B*Tp/s, k*C_in] x W2^T``
(`fk_gemm_nt`; TMA reads the overlapping rows straight from the padded signal -- no im2col copy, bias in the epilogue).  The rows
of a trial beyond its last output step mix in the next trial's padding and are sliced away.  The same view serves the backward:

* dW = dY^T A_view            (`fk_gemm_tn`, split-K over the B*T rows, deterministic)
* dX = the transposed convolution = the same kind of GEMM over the right-padded dY with the taps reversed; for the stride-2
  down-sampling conv (k = 4) both output parities come out of ONE GEMM with N = 2*C_in (row m = [dx[2m] | dx[2m+1]]).
* the stride-2 transposed convolution (k = 4, trailing k - s samples trimmed) likewise: y[2v + p] = x[v] W_p + x[v-1] W_{p+2},
  one 2-tap GEMM with N = 2*C_out whose output rows are [y[2v] | y[2v+1]].

All SoundStream convolutions have dilation 1 (vq_brain.py:48-63 builds every ResidualUnit with dilation 1).  No CPU path.

Streaming inference (`causal_conv1d_step`, used by SoundStream.stream) builds the same GEMM rows with the last k - 1 input
rows of the previous step in place of the causal zero padding (`fk_conv_stream_rows`, which also applies the ELU and the
ResidualUnit add that feed the convolution), so a step's outputs equal the offline ones row for row.
"""
from __future__ import annotations

import os

import torch

from . import gemm
from .ops import column_sum
from ._lib import FkError, check, lib, ptr, stream

BF16 = torch.bfloat16
PAD_IMPL = os.environ.get("FK_CONV_PAD", "own")      # "torch": zeros + strided copy (cross-check)


def _padded(x3: torch.Tensor, rows_per_trial: int, left: int, slack: int) -> torch.Tensor:
    """[B, T, C] -> flat bf16 buffer [(B * rows_per_trial + slack), C]: trial b occupies rows [b*rpt, (b+1)*rpt) with the data
    at offset `left`, zeros elsewhere (causal left padding, right padding, and `slack` rows so that the last im2col rows stay
    inside the allocation)."""
    B, T, C = x3.shape
    total = B * rows_per_trial + slack
    sb, st = (x3.stride(0), x3.stride(1)) if B > 1 else (T * x3.stride(1), x3.stride(1))
    if (PAD_IMPL == "own" and x3.dtype in (torch.float32, BF16) and C % 8 == 0 and x3.stride(2) == 1 and sb % 8 == 0 and st % 8 == 0
            and st >= C and x3.data_ptr() % 16 == 0 and B > 0 and T > 0 and x3.device.index == torch.cuda.current_device()):
        # one pass: zeros and data (fk_pad_rows); the autograd Functions below run on the tensors' device already
        buf = torch.empty(total, C, device=x3.device, dtype=BF16)
        check(lib().fk_pad_rows(ptr(x3), 0 if x3.dtype == torch.float32 else 1, B, T, C, sb, st, ptr(buf), rows_per_trial, left,
                                total, stream()), "fk_pad_rows")
        return buf
    buf = torch.zeros(total, C, device=x3.device, dtype=BF16)                            # (a memset, not a kernel)
    buf[:B * rows_per_trial].view(B, rows_per_trial, C)[:, left:left + T] = x3          # one copy, converts to bf16 on the way
    return buf


def _rows(buf: torch.Tensor, n_rows: int, taps: int, step: int) -> torch.Tensor:
    """im2col view: row m = buf[m*step : m*step + taps] flattened (overlapping rows, no copy)."""
    C = buf.shape[1]
    return torch.as_strided(buf, (n_rows, taps * C), (step * C, 1))


def _w_taps_major(weight: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, k] -> bf16 [Cout, k * Cin] (column = (tap, c_in)) in one permuting, converting copy."""
    Cout, Cin, k = weight.shape
    out = torch.empty(Cout, k * Cin, device=weight.device, dtype=BF16)
    out.view(Cout, k, Cin).copy_(weight.detach().permute(0, 2, 1))
    return out


def _w_transpose_pairs(weight: torch.Tensor, bias):
    """ConvTranspose1d (k = 4, stride 2) weight [Cin, Cout, 4] -> bf16 [2 Cout, 2 Cin] whose GEMM row v = [x[v-1] | x[v]]
    gives [y[2v] | y[2v+1]], and the bias doubled to match (fp32 [2 Cout], or None)."""
    wb = weight.detach().to(BF16)
    wt = [wb[:, :, j].t() for j in range(4)]                            # [Cout, Cin]
    w2 = torch.cat([torch.cat([wt[2], wt[0]], dim=1), torch.cat([wt[3], wt[1]], dim=1)], dim=0).contiguous()
    b2 = None if bias is None else torch.cat([bias.detach().float(), bias.detach().float()])
    return w2, b2


def conv_supported(c_in: int, c_out: int, k: int, stride: int, dilation: int = 1, groups: int = 1) -> bool:
    ok_shape = (c_in * k) % 64 == 0 and c_out % 64 == 0 and c_in % 8 == 0
    return dilation == 1 and groups == 1 and ok_shape and (stride == 1 or (stride == 2 and k == 4))


class _CausalConvFn(torch.autograd.Function):
    """y[b, t, :] = sum_j x[b, t*s + j - (k-1), :] W[:, :, j]^T + bias  (left padding k - 1, models/vq_brain.py:22-28)."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride):
        B, T, Cin = x.shape
        Cout, _, k = weight.shape
        s = stride
        T_out = (T - 1) // s + 1
        rpt = -(-(T + k - 1) // s) * s                                  # rows per trial, a multiple of the stride
        buf = _padded(x, rpt, k - 1, k)
        M = B * rpt // s
        A = _rows(buf, M, k, s)
        w2 = _w_taps_major(weight)                                      # [Cout, (tap, c_in)]
        y = gemm.gemm_nt(A, w2, bias, name="conv_fwd")
        ctx.save_for_backward(buf, weight)
        ctx.meta = (B, T, Cin, Cout, k, s, T_out, rpt, M, bias is not None, x.dtype)
        return y.view(B, rpt // s, Cout)[:, :T_out]

    @staticmethod
    def backward(ctx, g):
        buf, weight = ctx.saved_tensors
        B, T, Cin, Cout, k, s, T_out, rpt, M, has_bias, x_dtype = ctx.meta
        A = _rows(buf, M, k, s)
        # dY laid out like the output rows of the forward GEMM (zeros in the rows that were sliced away) + k slack rows
        gbuf = _padded(g, rpt // s, 0, k)
        g2 = gbuf[:M]
        dw = db = dx = None
        if ctx.needs_input_grad[1]:
            dw2 = gemm.gemm_tn(g2, A, name="conv_dw")                  # [Cout, k * Cin]
            dw = dw2.view(Cout, k, Cin).permute(0, 2, 1).to(weight.dtype).contiguous()        # (dense, as DDP's bucket views expect)
        if has_bias and ctx.needs_input_grad[2]:
            db = column_sum(g2)                                        # (the padded copy is contiguous; its extra rows are zero)
        if ctx.needs_input_grad[0]:
            if s == 1:
                # dx[u] = sum_j' g[u + j'] W_{k-1-j'}: im2col of the right-padded dY, taps reversed
                Ag = _rows(gbuf, M, k, 1)
                wd = torch.empty(Cin, k * Cout, device=g.device, dtype=BF16)
                wd.view(Cin, k, Cout).copy_(weight.detach().flip(2).permute(1, 2, 0))
                dx = gemm.gemm_nt(Ag, wd, None, name="conv_dx").view(B, rpt, Cin)[:, :T]
            else:
                # k = 4, s = 2: dx[2m] = g[m] W_3 + g[m+1] W_1, dx[2m+1] = g[m+1] W_2 + g[m+2] W_0 -> one GEMM, N = 2 Cin
                Ag = _rows(gbuf, M, 3, 1)
                wb = weight.detach().to(BF16)
                z = torch.zeros(Cin, Cout, device=g.device, dtype=BF16)
                wt = [wb[:, :, j].t() for j in range(4)]                # [Cin, Cout] each
                wd = torch.cat([torch.cat([wt[3], wt[1], z], dim=1), torch.cat([z, wt[2], wt[0]], dim=1)], dim=0).contiguous()
                dx = gemm.gemm_nt(Ag, wd, None, name="conv_dx").view(B, rpt // 2, 2 * Cin)[:, :T_out].reshape(B, 2 * T_out, Cin)[:, :T]
            if dx.dtype != x_dtype:
                dx = dx.to(x_dtype)
        return dx, dw, db, None


class _CausalConvTransposeFn(torch.autograd.Function):
    """conv_transpose1d(k = 4, stride 2) with the trailing k - s samples trimmed (models/vq_brain.py:31-45):
    y[b, 2v + p, :] = x[b, v, :] W[:, :, p] + x[b, v-1, :] W[:, :, p+2] + bias, weight [Cin, Cout, 4]."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        B, T, Cin = x.shape
        _, Cout, k = weight.shape
        rpt = T + 1
        buf = _padded(x, rpt, 1, 2)
        M = B * rpt
        A = _rows(buf, M, 2, 1)                                         # row v = [x[v-1] | x[v]]
        w2, b2 = _w_transpose_pairs(weight, bias)
        y = gemm.gemm_nt(A, w2, b2, name="convT_fwd")                   # row v = [y[2v] | y[2v+1]]
        ctx.save_for_backward(buf, weight)
        ctx.meta = (B, T, Cin, Cout, rpt, M, bias is not None, x.dtype)
        return y.view(B, rpt, 2 * Cout)[:, :T].reshape(B, 2 * T, Cout)

    @staticmethod
    def backward(ctx, g):
        buf, weight = ctx.saved_tensors
        B, T, Cin, Cout, rpt, M, has_bias, x_dtype = ctx.meta
        A = _rows(buf, M, 2, 1)
        gbuf = _padded(g.reshape(B, T, 2 * Cout), rpt, 0, 2)            # row v = [g[2v] | g[2v+1]], one zero row per trial
        g2 = gbuf[:M]
        dw = db = dx = None
        if ctx.needs_input_grad[1]:
            d = gemm.gemm_tn(g2, A, name="convT_dw")                    # [2 Cout, 2 Cin]: block (p, tap), tap 0 <-> W_{p+2}, tap 1 <-> W_p
            d = d.view(2, Cout, 2, Cin)
            dw = torch.stack([d[0, :, 1].t(), d[1, :, 1].t(), d[0, :, 0].t(), d[1, :, 0].t()], dim=2).to(weight.dtype)    # [Cin, Cout, 4] (dense)
        if has_bias and ctx.needs_input_grad[2]:
            db = column_sum(g2).view(2, Cout).sum(0)
        if ctx.needs_input_grad[0]:
            # dx[v] = [g[2v] | g[2v+1] | g[2v+2] | g[2v+3]] . [W_0 | W_1 | W_2 | W_3]
            Ag = _rows(gbuf, M, 2, 1)
            wd = _w_taps_major(weight)                                  # [Cin, (tap, c_out)]
            dx = gemm.gemm_nt(Ag, wd, None, name="convT_dx").view(B, rpt, Cin)[:, :T]
            if dx.dtype != x_dtype:
                dx = dx.to(x_dtype)
        return dx, dw, db


def _row_strides(x3: torch.Tensor):
    """(batch, token) strides in elements of a [B, T, C] operand; with B == 1 the batch stride is never used."""
    if x3.stride(2) != 1:
        raise FkError("streamed convolution operands must have contiguous channels")
    return (x3.stride(0), x3.stride(1)) if x3.shape[0] > 1 else (x3.shape[1] * x3.stride(1), x3.stride(1))


def causal_conv1d_step(x: torch.Tensor, r, elu: bool, hist_in, hist_out, w2: torch.Tensor, bias, taps: int, stride: int = 1,
                       counts=None):
    """One step of a streamed causal convolution (inference only): x [B, n, Cin] new rows (fp32 or bf16, row-strided), r
    (None or bf16 [B, n, Cin]) a residual added to x, `elu` the activation applied to x + r, hist_in / hist_out bf16
    [B, taps - 1, Cin] the last input rows of the previous step / of this one (None when taps == 1), w2 [Cout, taps * Cin]
    bf16 (`_w_taps_major`, or `_w_transpose_pairs` for the transposed convolution as 2 taps), bias fp32 or None.
    Returns (y bf16 [B, n / stride, Cout], the bf16 input rows act(x + r) [B, n, Cin] as a view of the GEMM operand).

    The GEMM rows are those of `_CausalConvFn.forward`, with the history in place of the causal zero padding.

    counts: optional device int32 [B], the new rows of each trial (0 ... n, multiples of the stride): rows past a trial's
    count are zeros in the GEMM input, so the outputs past counts[b] / stride are finite whatever x holds there, and the
    history advances by counts[b] rows only."""
    B, n, Cin = x.shape
    h, s = taps - 1, stride
    if n % s != 0:
        raise FkError(f"causal_conv1d_step: {n} rows is not a multiple of the stride {s}")
    if (hist_in is None) != (h == 0) or (h > 0 and (hist_in.shape != (B, h, Cin) or hist_out.shape != (B, h, Cin))):
        raise FkError(f"causal_conv1d_step: the history must be [{B}, {h}, {Cin}]")
    rpt = -(-(n + h) // s) * s                                          # rows per trial, a multiple of the stride
    total = B * rpt + taps
    buf = torch.empty(total, Cin, device=x.device, dtype=BF16)
    rs = (0, 0) if r is None else _row_strides(r)
    check(lib().fk_conv_stream_rows_counts(ptr(x), 0 if x.dtype == torch.float32 else 1, *_row_strides(x), ptr(r), *rs,
                                           ptr(hist_in), ptr(hist_out), ptr(counts), B, n, h, Cin, int(elu), ptr(buf), rpt, total,
                                           stream()),
          "fk_conv_stream_rows")
    M = B * rpt // s
    y = gemm.gemm_nt(_rows(buf, M, taps, s), w2, bias, name="conv_stream")
    return y.view(B, rpt // s, w2.shape[0])[:, :n // s], buf[:B * rpt].view(B, rpt, Cin)[:, h:h + n]


def causal_conv1d_cl(x: torch.Tensor, weight: torch.Tensor, bias, stride: int = 1) -> torch.Tensor:
    """channels-last causal Conv1d: x [B, T, Cin], weight [Cout, Cin, k] (nn.Conv1d layout) -> bf16 [B, T/stride, Cout]."""
    if not x.is_cuda:
        raise FkError("frankenstein_b200 kernels run on a B200 only (no CPU fallback)")
    return _CausalConvFn.apply(x, weight, bias, stride)


def causal_conv_transpose1d_cl(x: torch.Tensor, weight: torch.Tensor, bias) -> torch.Tensor:
    """channels-last causal ConvTranspose1d (k = 4, stride 2, trimmed): x [B, T, Cin], weight [Cin, Cout, 4] -> bf16 [B, 2T, Cout]."""
    if not x.is_cuda:
        raise FkError("frankenstein_b200 kernels run on a B200 only (no CPU fallback)")
    if weight.shape[2] != 4:
        raise FkError("causal_conv_transpose1d_cl is built for kernel size 4, stride 2")
    return _CausalConvTransposeFn.apply(x, weight, bias)
