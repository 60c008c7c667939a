"""Dense projections of the transformer blocks on the library's own tcgen05 GEMM kernels (csrc/gemm.cu).

Functional wrappers (``gemm_nt``, ``gemm_tn``) and the ``torch.autograd.Function``s the modules use:

* ``linear``       -- ``nn.Linear`` (models/brainformer.py:171 ``project``, ``to_signals``, ...): y = x W^T (+ b);
* ``qkv_rope``     -- qw / kw / vw as ONE projection (brainformer.py:141-143) with ``apply_rope`` (:70-91, :156-158) applied
                      to the q | k columns in the GEMM epilogue (heads of 16, 32 or 64 columns);
* ``swiglu_mlp``   -- ``w2(silu(w1 x) * w3 x)`` (brainformer.py:119-124): the w1 | w3 projection forms the gate in its
                      epilogue; the backward applies the SwiGLU derivative in one streaming pass after the d-gated GEMM.

Weights stay fp32 ``nn.Parameter``s under their reference names; each call casts them to bf16 (and, for the input
gradient, makes the transposed copy the NT kernel wants -- a few MB).  Weight gradients come from ``fk_gemm_tn``
(dW = dY^T X, contraction over the tokens, fixed-order split reduction: bit-reproducible).  CPU tensors raise.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

from ._lib import FkError, check, lib, on_tensor_device, ptr, require_cuda, require_device, stream, timed

BF16 = torch.bfloat16
EPI_STORE, EPI_ROPE, EPI_SWIGLU, EPI_ROPE64, EPI_ROPE16 = 0, 1, 2, 4, 5
# head width -> RoPE epilogue of the fused q | k | v projection
ROPE_EPILOGUE = {16: EPI_ROPE16, 32: EPI_ROPE, 64: EPI_ROPE64}
ROPE_EPILOGUES = tuple(ROPE_EPILOGUE.values())


def _as2d(x: torch.Tensor) -> torch.Tensor:
    x2 = x.reshape(-1, x.shape[-1])
    if x2.dtype != BF16:
        x2 = x2.to(BF16)
    if x2.stride(-1) != 1 or x2.stride(0) % 8 != 0 or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    return x2


@on_tensor_device
def gemm_nt(a: torch.Tensor, b: torch.Tensor, bias: Optional[torch.Tensor] = None, epilogue: int = EPI_STORE, *,
            rope=None, rope_cols: int = 0, rope_S: int = 0, lead: Optional[tuple] = None, name: str = "gemm_nt"):
    """C [M, N] bf16 = a [M, K] @ b [N, K]^T on tcgen05 (fp32 accumulate).  See include/fk_b200.h (fk_gemm_nt) for the
    epilogues.  Returns C (EPI_STORE / EPI_ROPE / EPI_ROPE64 / EPI_ROPE16) or (h13, gated) (EPI_SWIGLU).
    lead (EPI_STORE): C is allocated as [*lead, N] (prod(lead) = M), a tensor of its own rather than a view of [M, N]."""
    require_cuda(a, b)
    require_device()
    if a.dtype != BF16 or b.dtype != BF16:
        raise FkError("gemm_nt expects bf16 operands")
    M, K = a.shape
    N = b.shape[0]
    if b.shape[1] != K:
        raise FkError(f"gemm_nt: inner dimensions differ ({tuple(a.shape)} x {tuple(b.shape)}^T)")
    if a.stride(1) != 1 or b.stride(1) != 1:
        raise FkError("gemm_nt: operands must be row-major")
    dev = a.device
    C = C2 = None
    ldc = ldc2 = 0
    if lead is not None and (epilogue != EPI_STORE or math.prod(lead) != M):
        raise FkError(f"gemm_nt: output shape {(*lead, N)} does not hold [{M}, {N}]")
    if epilogue == EPI_STORE or epilogue in ROPE_EPILOGUES:
        C = torch.empty(*(lead if lead is not None else (M,)), N, device=dev, dtype=BF16)
        ldc = N
    elif epilogue == EPI_SWIGLU:
        C = torch.empty(M, N, device=dev, dtype=BF16)
        C2 = torch.empty(M, N // 2, device=dev, dtype=BF16)
        ldc, ldc2 = N, N // 2
    bias_f = None
    if bias is not None:
        bias_f = bias.detach().float().contiguous()
    table, pos, rope_len, rope_off = None, None, 0, 0
    if epilogue in ROPE_EPILOGUES:
        table, pos, rope_len, rope_off = rope.table, rope.pos, rope.table.shape[0], rope.offset
        if pos is not None:
            pos = pos.reshape(-1)
            if pos.numel() != M:
                raise FkError("gemm_nt: rope positions must cover every row")
    with timed(name, 2.0 * M * N * K):
        check(lib().fk_gemm_nt(ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(C), ldc, M, N, K, ptr(bias_f), epilogue,
                               ptr(C2), ldc2, ptr(table), rope_len, ptr(pos), rope_off, rope_cols, rope_S, stream()),
              "fk_gemm_nt")
    if epilogue == EPI_SWIGLU:
        return C, C2
    return C


@on_tensor_device
def gemm_tn(a: torch.Tensor, b: torch.Tensor, name: str = "gemm_tn") -> torch.Tensor:
    """out [Na, Nb] fp32 = a [M, Na]^T @ b [M, Nb] (bf16 row-major operands): the weight gradient of a Linear."""
    require_cuda(a, b)
    require_device()
    if a.dtype != BF16 or b.dtype != BF16 or a.stride(1) != 1 or b.stride(1) != 1 or a.shape[0] != b.shape[0]:
        raise FkError("gemm_tn expects row-major bf16 operands with the same number of rows")
    M, Na = a.shape
    Nb = b.shape[1]
    splits = lib().fk_gemm_tn_splits(M, Na, Nb, 0)
    out = torch.empty(Na, Nb, device=a.device, dtype=torch.float32)
    ws = torch.empty(splits, Na, Nb, device=a.device, dtype=torch.float32)
    with timed(name, 2.0 * M * Na * Nb):
        check(lib().fk_gemm_tn(ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(out), M, Na, Nb, ptr(ws), splits, stream()),
              "fk_gemm_tn")
    return out


def nt_ok(K: int, N: int) -> bool:
    return K % 8 == 0 and N % 32 == 0


def tn_ok(Na: int, Nb: int) -> bool:
    return Na % 64 == 0 and Nb % 64 == 0


# ------------------------------------------------------------------------------------------------
# nn.Linear
# ------------------------------------------------------------------------------------------------
class _LinearFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, x, weight, bias):
        x2 = _as2d(x)
        wb = weight.detach().to(BF16).contiguous()
        # y is allocated in x's leading shape rather than returned as a view: attention_qkv rotates q and k of a fused
        # q | k | v projection in place, which autograd refuses on a view
        y = gemm_nt(x2, wb, bias, EPI_STORE, lead=tuple(x.shape[:-1]), name="gemm_linear")
        ctx.save_for_backward(x2, wb)
        ctx.in_shape, ctx.in_dtype, ctx.w_dtype = x.shape, x.dtype, weight.dtype
        ctx.has_bias = bias is not None
        ctx.b_dtype = bias.dtype if bias is not None else None
        return y

    @staticmethod
    @on_tensor_device
    def backward(ctx, gy):
        x2, wb = ctx.saved_tensors
        g2 = _as2d(gy)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = gemm_nt(g2, wb.t().contiguous(), None, EPI_STORE, name="gemm_linear_dx").view(ctx.in_shape)
            if dx.dtype != ctx.in_dtype and ctx.in_dtype in (torch.float32, torch.float16):
                dx = dx.to(ctx.in_dtype)
        if ctx.needs_input_grad[1]:
            dw = gemm_tn(g2, x2, name="gemm_linear_dw").to(ctx.w_dtype)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            from .ops import column_sum                 # (ops imports nothing from this module at import time)
            db = column_sum(g2).to(ctx.b_dtype)
        return dx, dw, db


def linear_supported(in_features: int, out_features: int) -> bool:
    """forward (NT, K = in), input gradient (NT, K = out) and weight gradient (TN) shapes all fit the kernels."""
    return (nt_ok(in_features, out_features) and nt_ok(out_features, in_features) and tn_ok(out_features, in_features))


def linear(x, weight, bias=None):
    """y = x W^T (+ b) in bf16 on the library's GEMM (fp32 accumulate); x [..., K], W [N, K]."""
    return _LinearFn.apply(x, weight, bias)


# ------------------------------------------------------------------------------------------------
# fused q | k | v projection with RoPE
# ------------------------------------------------------------------------------------------------
class _QKVRopeFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, x, wq, wk, wv, rope, n_heads):
        B, S, _ = x.shape
        x2 = _as2d(x)
        w = torch.cat([wq.detach(), wk.detach(), wv.detach()], dim=0).to(BF16)
        inner = wq.shape[0]
        if rope is not None:
            epi = ROPE_EPILOGUE.get(inner // n_heads)
            if epi is None:
                raise FkError(f"qkv_rope: the RoPE epilogue takes heads of 16, 32 or 64 columns, not {inner // n_heads}")
            qkv = gemm_nt(x2, w, None, epi, rope=rope, rope_cols=2 * inner, rope_S=S, name="gemm_qkv_rope")
        else:
            qkv = gemm_nt(x2, w, None, EPI_STORE, name="gemm_qkv_rope")
        ctx.save_for_backward(x2, w)
        ctx.in_shape, ctx.in_dtype, ctx.w_dtype, ctx.inner = x.shape, x.dtype, wq.dtype, inner
        return qkv.view(B, S, 3 * inner)

    @staticmethod
    @on_tensor_device
    def backward(ctx, g):
        # g: gradient w.r.t. the (pre-rotation) projection -- the attention backward has already rotated dq / dk back
        x2, w = ctx.saved_tensors
        g2 = _as2d(g)
        dx = gemm_nt(g2, w.t().contiguous(), None, EPI_STORE, name="gemm_qkv_dx").view(ctx.in_shape)
        if dx.dtype != ctx.in_dtype and ctx.in_dtype in (torch.float32, torch.float16):
            dx = dx.to(ctx.in_dtype)
        dw = gemm_tn(g2, x2, name="gemm_qkv_dw").to(ctx.w_dtype)
        i = ctx.inner
        return dx, dw[:i], dw[i:2 * i], dw[2 * i:], None, None


def qkv_supported(dim: int, inner: int) -> bool:
    return dim <= 512 and nt_ok(dim, 3 * inner) and nt_ok(3 * inner, dim) and tn_ok(3 * inner, dim) and inner % 32 == 0


def qkv_rope(x, wq, wk, wv, rope, n_heads):
    """[B, S, dim] -> fused [B, S, 3 * inner] bf16 projection (q | k | v) with q and k already rotated."""
    return _QKVRopeFn.apply(x, wq, wk, wv, rope, n_heads)


# ------------------------------------------------------------------------------------------------
# SwiGLU MLP
# ------------------------------------------------------------------------------------------------
def _interleave(w1, w3):
    """[w1[0:128]; w3[0:128]; w1[128:256]; w3[128:256]; ...]: every 256-column tile of the fused projection holds the
    w1 and the w3 outputs of the same 128 hidden units, so the gate is formed inside one epilogue tile."""
    H, D = w1.shape
    return torch.stack([w1.view(H // 128, 128, D), w3.view(H // 128, 128, D)], dim=1).reshape(2 * H, D)


def _deinterleave(w13):
    H2, D = w13.shape
    v = w13.view(H2 // 256, 2, 128, D)
    return v[:, 0].reshape(H2 // 2, D), v[:, 1].reshape(H2 // 2, D)


class _SwiGLUMLPFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, x, w1, w3, w2):
        x2 = _as2d(x)
        w13 = _interleave(w1.detach(), w3.detach()).to(BF16)
        w2b = w2.detach().to(BF16).contiguous()
        h13, gated = gemm_nt(x2, w13, None, EPI_SWIGLU, name="gemm_w13_swiglu")
        out = gemm_nt(gated, w2b, None, EPI_STORE, name="gemm_w2")
        ctx.save_for_backward(x2, h13, gated, w13, w2b)
        ctx.in_shape, ctx.in_dtype, ctx.w_dtype = x.shape, x.dtype, w1.dtype
        return out.view(*x.shape[:-1], w2.shape[0])

    @staticmethod
    @on_tensor_device
    def backward(ctx, g):
        x2, h13, gated, w13, w2b = ctx.saved_tensors
        g2 = _as2d(g)
        # d gated on the plain epilogue, then the SwiGLU derivative as one HBM-bound pass over h13 / dh13: the pass is
        # bound by the 8.6 GB it moves either way, and the streaming kernel keeps more bytes in flight than a GEMM
        # epilogue can (measured: 1.2 + 1.5 ms against 4.4 ms with the derivative in the epilogue at M = 524288)
        dg = gemm_nt(g2, w2b.t().contiguous(), None, EPI_STORE, name="gemm_dgated")
        dh13 = torch.empty_like(h13)
        M, H = dg.shape
        with timed("swiglu_bwd", 0.0):
            check(lib().fk_swiglu_backward_blocked(ptr(h13), ptr(dg), ptr(dh13), M, H, 128, stream()),
                  "fk_swiglu_backward_blocked")
        del dg
        dw2 = gemm_tn(g2, gated, name="gemm_w2_dw").to(ctx.w_dtype)
        dx = gemm_nt(dh13, w13.t().contiguous(), None, EPI_STORE, name="gemm_w13_dx").view(ctx.in_shape)
        if dx.dtype != ctx.in_dtype and ctx.in_dtype in (torch.float32, torch.float16):
            dx = dx.to(ctx.in_dtype)
        dw1, dw3 = _deinterleave(gemm_tn(dh13, x2, name="gemm_w13_dw"))
        return dx, dw1.to(ctx.w_dtype), dw3.to(ctx.w_dtype), dw2


def mlp_supported(dim: int, hidden: int) -> bool:
    return (dim <= 512 and dim % 64 == 0 and hidden % 128 == 0)


def swiglu_mlp(x, w1, w3, w2):
    """w2(silu(w1 x) * (w3 x)) with the gate fused into the w1 | w3 projection (forward); the backward applies its
    derivative in one streaming pass after the d-gated GEMM."""
    return _SwiGLUMLPFn.apply(x, w1, w3, w2)


# ------------------------------------------------------------------------------------------------
# patch embedding (brainformer.Encoder: to_patches + Linear(patch -> dim) + bias)
# ------------------------------------------------------------------------------------------------
def patch_embed_supported(T: int, E: int, patch: int, dim: int) -> bool:
    return patch in (16, 32, 48, 64) and T % patch == 0 and E % 64 == 0 and dim % 64 == 0


class _PatchEmbedFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, x, weight, bias):
        require_cuda(x, weight)
        require_device()
        B, T, E = x.shape
        dim, patch = weight.shape
        xb = x.detach().to(BF16).contiguous().view(B * T, E)
        wt = weight.detach().t().contiguous().to(BF16)                      # W^T [patch, dim]
        bias_f = None if bias is None else bias.detach().float().contiguous()
        out = torch.empty(B, (T // patch) * E, dim, device=x.device, dtype=BF16)
        with timed("gemm_patch_embed", 2.0 * B * T * E * dim):
            check(lib().fk_patch_embed_forward(ptr(xb), E, ptr(wt), ptr(bias_f), None, ptr(out), B * T, E, patch, dim, stream()),
                  "fk_patch_embed_forward")
        ctx.save_for_backward(xb)
        ctx.meta = (B, T, E, patch, dim, weight.dtype, None if bias is None else bias.dtype)
        return out

    @staticmethod
    @on_tensor_device
    def backward(ctx, g):
        (xb,) = ctx.saved_tensors
        B, T, E, patch, dim, w_dtype, b_dtype = ctx.meta
        M = B * (T // patch) * E
        g2 = _as2d(g)
        # dW[n, k] = sum over tokens g[token, n] * patch[token, k], db[n] = sum g[token, n]: ONE split-K TN product against
        # [patches | 1 | 0 ...] (the patch matrix exists only here, 64 bf16 columns per token, never in the forward pass)
        cols = 64 if patch < 64 else 128
        ext = torch.zeros(M, cols, device=g.device, dtype=BF16)
        ext[:, :patch] = xb.view(B, T // patch, patch, E).transpose(2, 3).reshape(M, patch)
        ext[:, patch] = 1.0
        dwb = gemm_tn(g2, ext, name="gemm_patch_embed_dw")                  # [dim, cols] fp32
        dw = dwb[:, :patch].to(w_dtype)
        db = None if b_dtype is None else dwb[:, patch].to(b_dtype)
        return None, dw, db


def patch_embed(x, weight, bias=None):
    """[B, T, E] signal -> [B, (T/p) * E, dim] bf16 tokens, token = (time patch, electrode), = Linear(p -> dim)(to_patches(x))
    (models/brainformer.py:282-285) without materialising the patch tensor.  x gets no gradient (it is data)."""
    if x.requires_grad:
        raise FkError("patch_embed: the input signal is data (no input gradient); use Encoder.embed(to_patches(x)) otherwise")
    return _PatchEmbedFn.apply(x, weight, bias)
