"""Brainformer -- host-side mirror of the reference ``models/brainformer.py``.

Same public names, constructor arguments, ``forward`` signatures and state-dict keys as the reference
(models/brainformer.py:17-574), so ``Encoder``, ``MAE``, ``BrainFormer``, ``CrossBlock``, ``Config`` ... drop
into ``notebooks_trainer/{train_mae,train_brainformer,franky_baseline_gpt2}.ipynb`` and
``utils/train_utils.py:138``.  What runs underneath (bf16 compute, fp32 accumulate, fp32 residual stream and
fp32 master weights):

* LayerNorm / RMSNorm, SwiGLU gate, RoPE: fused bandwidth-bound kernels (``ops.py`` -> libfk_b200.so);
* self-attention (head_dim 16, 32 or 64): flash-style kernel with the block-causal / gathered / padding mask
  evaluated analytically from integer labels -- the ``[S,S]`` (or ``[B,1,s,s]``) bool masks of the reference
  are never read (``attn_mask`` stays a registered buffer only so checkpoints keep their keys);
* q/k/v as ONE fused projection (weights stay three ``nn.Linear`` modules for checkpoint compatibility),
  w1/w3 as one fused projection; the dense GEMMs themselves are cuBLAS library calls.

Callers that pass the reference's dense mask / complex rope tensors to ``Block`` directly (e.g. the notebook's
``BrainEncoder`` with ``CrossBlock``) are served by a compatibility path on library SDPA; the perceiver
(head_dim 16, <= 32 queries) is SURVEY section 8a row a9 "keep torch ops".
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

import os

from . import gemm, ops
from .ops import LabelMask, RopeSpec

# "own" (default): the dense projections run on the library's tcgen05 GEMMs with fused epilogues (csrc/gemm.cu);
# "cublas": the same math through F.linear + the separate RoPE / SwiGLU kernels (A/B comparison only).
GEMM_IMPL = os.environ.get("FK_GEMM", "own")

try:  # the reference derives its configs from simple_parsing's Serializable; optional here
    from simple_parsing.helpers import Serializable as _ConfigBase
except Exception:  # pragma: no cover - simple_parsing is not installed in the build image
    class _ConfigBase:
        pass

BF16 = torch.bfloat16
_INT32_MAX = 2 ** 31 - 1


@dataclass
class MAEConfig(_ConfigBase):
    """models/brainformer.py:17-38 (same fields and defaults)."""
    window_size: int = 1024
    n_electrodes: int = 256
    patch_size: int = 48
    dim: int = 256
    n_layers: int = 4
    head_dim: int = 32
    hidden_dim: int = 1024
    n_heads: int = 8
    n_kv_heads: int = 8
    rope_theta: int = 10000
    n_dec_layers: Optional[int] = 4
    decoder_dim: Optional[int] = 256


@dataclass
class Config(_ConfigBase):
    """models/brainformer.py:40-53 (same fields and defaults)."""
    encoder: MAEConfig
    n_output_tokens: int = 32
    output_dim: int = 1024
    dim: int = 256
    n_layers: int = 2
    head_dim: int = 16
    hidden_dim: int = 512
    n_heads: int = 4
    n_kv_heads: int = 4
    rope_theta: int = 10_000


def rope_inv_freq(dim: int, theta: float) -> torch.Tensor:
    """fp32 [dim//2] theta^(-2j/dim), the RoPE frequencies of build_complex_rope_cache."""
    return 1.0 / (theta ** (torch.arange(0, dim, 2).float() / dim))


def build_complex_rope_cache(dim: int, seq_len: int, theta: float) -> torch.Tensor:
    """[seq_len, dim//2] complex64 unit phasors exp(i * t * theta^(-2j/dim))  (models/brainformer.py:56-68)."""
    inv_freq = rope_inv_freq(dim, theta)
    angles = torch.outer(torch.arange(seq_len), inv_freq).float()
    return torch.polar(torch.ones_like(angles), angles)


def apply_rope(x: torch.Tensor, rope: torch.Tensor):
    """Library restatement of models/brainformer.py:70-91 for callers that hold complex rope tensors."""
    T = x.size(1)
    rope = rope[-T:] if rope.dim() == 2 else rope[:, -T:]
    xc = torch.view_as_complex(x.float().reshape(*x.shape[:-1], -1, 2))
    return torch.view_as_real(xc * rope.unsqueeze(-2)).flatten(3).type_as(x)


def build_advanced_causal_mask(block_size, tok_per_time):
    """bool [block_size, block_size], True = attend: causal at the granularity of tok_per_time-token groups
    (models/brainformer.py:93-111).  Built from the label rule the attention kernel evaluates."""
    blk = torch.arange(block_size) // tok_per_time
    return blk[None, :] <= blk[:, None]


def _linear_bf16(x, weight, bias=None):
    """bf16 GEMM regardless of the caller's autocast dtype: the reference trainer runs fp16 autocast
    (utils/train_utils.py:96), under which F.linear would re-cast the bf16 operands to fp16 and hand fp16 activations to
    kernels that take bf16.  The compute dtype of this package is bf16 (fp32 accumulate) whatever autocast says."""
    if GEMM_IMPL == "own" and x.is_cuda and gemm.linear_supported(weight.shape[1], weight.shape[0]):
        return gemm.linear(x, weight, bias)
    # shapes outside the kernels' granularity (e.g. the 32-wide patch projections) stay on the library GEMM
    with torch.autocast("cuda", enabled=False):
        return F.linear(x.to(BF16), weight.to(BF16), None if bias is None else bias.to(BF16))


class MLP(nn.Module):
    """w2(silu(w1 x) * w3 x)  (models/brainformer.py:115-124)."""

    def __init__(self, config):
        super().__init__()
        self.w1 = nn.Linear(config.dim, config.hidden_dim, bias=False)
        self.w2 = nn.Linear(config.hidden_dim, config.dim, bias=False)
        self.w3 = nn.Linear(config.dim, config.hidden_dim, bias=False)

    def forward(self, x) -> torch.Tensor:
        if not x.is_cuda:
            raise ops.FkError("frankenstein_b200 modules run on a B200 only (no CPU fallback)")
        hidden, dim = self.w1.weight.shape
        if GEMM_IMPL == "own" and gemm.mlp_supported(dim, hidden):
            # w1 | w3 as one tcgen05 GEMM whose epilogue forms the gate; backward fuses the SwiGLU derivative likewise
            return gemm.swiglu_mlp(x, self.w1.weight, self.w3.weight, self.w2.weight)
        w13 = torch.cat([self.w1.weight, self.w3.weight], dim=0)
        gated = ops.swiglu(_linear_bf16(x, w13))
        return _linear_bf16(gated, self.w2.weight)


def _dense_mask_attention(q, k, v, attn_mask):
    """compatibility path: the caller handed a dense bool mask (reference convention)."""
    if attn_mask is not None:
        attn_mask = attn_mask[..., -q.size(2):, -k.size(2):]
    return F.scaled_dot_product_attention(q, k, v, attn_mask=attn_mask)


class CausalSelfAttention(nn.Module):
    """models/brainformer.py:126-173.  attn_mask: LabelMask | dense bool tensor | None; rope: RopeSpec |
    complex tensor | None."""

    def __init__(self, config, is_causal=True):
        super().__init__()
        assert config.n_heads == config.n_kv_heads, "n_heads should be equal n_kv_heads"
        self.n_heads = config.n_heads
        self.n_kv_heads = config.n_heads
        self.repeats = 1
        self.head_dim = config.head_dim
        inner = config.head_dim * config.n_heads
        self.qw = nn.Linear(config.dim, inner, bias=False)
        self.kw = nn.Linear(config.dim, inner, bias=False)
        self.vw = nn.Linear(config.dim, inner, bias=False)
        self.project = nn.Linear(inner, config.dim, bias=False)

    def forward(self, x, attn_mask, rope, kv_cache=None):
        if not x.is_cuda:
            raise ops.FkError("frankenstein_b200 modules run on a B200 only (no CPU fallback)")
        B, T, _ = x.shape
        spec = rope
        if isinstance(rope, torch.Tensor) and rope.dim() == 2 and self.head_dim in (16, 32, 64):
            spec = RopeSpec.from_complex(rope, T, last=True)           # reference convention: rope[-T:]
        # unmasked calls with few tokens at head_dim != 32 (the perceiver's self-attention Block) take the few-query kernel
        small_ok = (attn_mask is None and self.head_dim != 32 and ops.small_attention_supported(T, self.head_dim)
                    and (rope is None or (isinstance(rope, torch.Tensor) and rope.dim() == 2)))
        kernel_ok = (self.head_dim in (16, 32, 64) and not small_ok and (attn_mask is None or isinstance(attn_mask, LabelMask))
                     and (spec is None or isinstance(spec, RopeSpec)))
        inner, dim = self.qw.weight.shape
        if kernel_ok and GEMM_IMPL == "own" and gemm.qkv_supported(dim, inner):
            # one tcgen05 GEMM for q | k | v with RoPE applied to q and k in its epilogue (no separate rope pass)
            qkv = gemm.qkv_rope(x, self.qw.weight, self.kw.weight, self.vw.weight, spec, self.n_heads)
            res = ops.attention_qkv(qkv, self.n_heads, spec, attn_mask, rope_applied=True)
            return _linear_bf16(res, self.project.weight)
        wqkv = torch.cat([self.qw.weight, self.kw.weight, self.vw.weight], dim=0)
        qkv = _linear_bf16(x, wqkv)
        if kernel_ok:
            res = ops.attention_qkv(qkv, self.n_heads, spec, attn_mask)
        elif small_ok:
            # the perceiver's self-attention Block (<= 64 tokens, head_dim 16): RoPE applied on load inside the kernel
            rs = None if rope is None else RopeSpec.from_complex(rope, T, last=True)       # reference convention: rope[-T:]
            q, k, v = qkv.view(B, T, 3, inner).unbind(2)
            res = ops.small_attention(q, k, v, self.n_heads, rope=rs)
        else:
            q, k, v = qkv.view(B, T, 3, self.n_heads, self.head_dim).unbind(2)
            if isinstance(rope, RopeSpec):
                raise ops.FkError("RopeSpec needs the head_dim-16 / 32 / 64 kernel path")
            if rope is not None:
                q, k = apply_rope(q, rope), apply_rope(k, rope)
            if isinstance(attn_mask, LabelMask):
                attn_mask = attn_mask.dense()
            res = _dense_mask_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), attn_mask)
            res = res.transpose(1, 2).reshape(B, T, self.n_heads * self.head_dim)
        return _linear_bf16(res, self.project.weight)


class CausalCrossAttention(nn.Module):
    """models/brainformer.py:175-219 (perceiver resampler, SURVEY 8a row a9 / 8f row N2): a few learnable queries against the
    whole token sequence -> the split-key kernels of csrc/small_attention.cu; dense-mask SDPA only for shapes outside them."""

    def __init__(self, config, is_causal=True):
        super().__init__()
        assert config.n_heads == config.n_kv_heads, "n_heads should be equal n_kv_heads"
        self.n_heads = config.n_heads
        self.n_kv_heads = config.n_heads
        self.repeats = 1
        inner = config.head_dim * config.n_heads
        self.qw = nn.Linear(config.dim, inner, bias=False)
        self.kw = nn.Linear(config.dim, inner, bias=False)
        self.vw = nn.Linear(config.dim, inner, bias=False)
        self.project = nn.Linear(inner, config.dim, bias=False)
        self.kv_cache = None

    def forward(self, x, context, attn_mask=None, use_kv_cache=None):
        B, T, _ = x.shape
        S = context.shape[1]
        q = _linear_bf16(x, self.qw.weight)
        ctx_bf16 = context.to(BF16)
        hd = q.shape[-1] // self.n_heads
        if attn_mask is None and x.is_cuda and ops.small_attention_supported(T, hd):
            # few learnable queries against thousands of context tokens: the split-key kernel of csrc/small_attention.cu,
            # fed by ONE fused k | v projection that it reads in place and whose gradient it writes as one buffer (one pass
            # over the context per GEMM instead of two, no gradient add of the two context gradients)
            kv = _linear_bf16(ctx_bf16, torch.cat([self.kw.weight, self.vw.weight], dim=0))
            res = ops.small_attention_kv(q, kv, self.n_heads)
        else:
            # two projections: slicing a fused buffer costs a zero-fill + strided copy per slice in autograd (select_backward)
            k = _linear_bf16(ctx_bf16, self.kw.weight)
            v = _linear_bf16(ctx_bf16, self.vw.weight)
            q, k, v = (t.view(B, t.shape[1], self.n_heads, -1).transpose(1, 2) for t in (q, k, v))
            res = _dense_mask_attention(q, k, v, attn_mask)
            res = res.transpose(1, 2).reshape(B, T, -1)
        return _linear_bf16(res, self.project.weight)


class RMSNorm(torch.nn.Module):
    """models/brainformer.py:221-232."""

    def __init__(self, dim: int, eps: float = 1e-6):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(dim))

    def forward(self, x, out_dtype=None):
        return ops.rms_norm(x, self.weight, self.eps, out_dtype or (x.dtype if x.dtype in (torch.float32, BF16) else torch.float32))


class _KernelLayerNorm(nn.LayerNorm):
    """nn.LayerNorm parameters (same state-dict keys), fused fp32-statistics kernel; emits bf16 for the GEMM
    that follows unless told otherwise."""

    def forward(self, x, out_dtype=BF16):
        if not x.is_cuda:
            raise ops.FkError("frankenstein_b200 modules run on a B200 only (no CPU fallback)")
        return ops.layer_norm(x, self.weight, self.bias, self.eps, out_dtype)


class Block(nn.Module):
    """pre-LN transformer block  (models/brainformer.py:234-245)."""

    def __init__(self, config):
        super().__init__()
        self.ln_1 = _KernelLayerNorm(config.dim)
        self.attn = CausalSelfAttention(config)
        self.ln_2 = _KernelLayerNorm(config.dim)
        self.mlp = MLP(config)

    def forward(self, x, attn_mask=None, rope=None, kv_cache=False):
        x = x + self.attn(self.ln_1(x), attn_mask, rope, kv_cache=kv_cache)
        x = x + self.mlp(self.ln_2(x))
        return x


def run_blocks(blocks, h, attn_mask=None, rope=None, final_norm=None, final_dtype=torch.float32, h_delta=None):
    """A stack of pre-LN Blocks on the fp32 residual stream `h` with every `x = x + branch` fused into the LayerNorm
    that follows it (ops.add_layer_norm): identical math to calling the Blocks one after another
    (models/brainformer.py:242-245, 345-351), one pass over the residual stream per add+norm instead of three.
    Returns (h, y) where y = final_norm(h) if final_norm is given, else None.
    h_delta (bf16): the stream starts as h + h_delta with h [1, S, D] broadcast over the batch (embedding table +
    patch projection, brainformer.py:343); the sum is formed inside the first fused add+LayerNorm."""
    n = len(blocks)
    if h_delta is not None and not (n > 0 and h.dtype == torch.float32 and isinstance(blocks[0].ln_1, _KernelLayerNorm)):
        h, h_delta = h_delta.float() + h, None
    if n == 0:
        return h, (final_norm(h, out_dtype=final_dtype) if final_norm is not None else None)
    if h.dtype != torch.float32 or not isinstance(blocks[0].ln_1, _KernelLayerNorm):
        for blk in blocks:                                   # generic path (e.g. RMSNorm blocks, bf16 streams)
            h = blk(h, attn_mask=attn_mask, rope=rope)
        return h, (final_norm(h, out_dtype=final_dtype) if final_norm is not None else None)
    if h_delta is not None:
        l0 = blocks[0].ln_1
        h, y = ops.add_layer_norm(h, h_delta, l0.weight, l0.bias, l0.eps)
    else:
        y = blocks[0].ln_1(h)
    for i, blk in enumerate(blocks):
        a = blk.attn(y, attn_mask, rope)
        h, y = ops.add_layer_norm(h, a, blk.ln_2.weight, blk.ln_2.bias, blk.ln_2.eps)
        m = blk.mlp(y)
        if i + 1 < n:
            nxt = blocks[i + 1].ln_1
            h, y = ops.add_layer_norm(h, m, nxt.weight, nxt.bias, nxt.eps)
        elif final_norm is not None:
            h, y = ops.add_layer_norm(h, m, final_norm.weight, final_norm.bias, final_norm.eps, final_dtype)
        else:
            h, y = h + m, None
    return h, y


class CrossBlock(nn.Module):
    """cross-attention + MLP, then a self-attention Block  (models/brainformer.py:247-268)."""

    def __init__(self, config):
        super().__init__()
        self.sa_block = Block(config)
        self.ln_1 = _KernelLayerNorm(config.dim)
        self.cross_attn = CausalCrossAttention(config)
        self.ln_2 = _KernelLayerNorm(config.dim)
        self.mlp = MLP(config)

    def forward(self, x, context, self_attn_mask=None, cross_attn_mask=None, sa_rope=None):
        x = x + self.cross_attn(self.ln_1(x), context, attn_mask=cross_attn_mask)
        x = x + self.mlp(self.ln_2(x))
        return self.sa_block(x, attn_mask=self_attn_mask, rope=sa_rope)


class Encoder(nn.Module):
    """models/brainformer.py:271-352.  x [B, T, n_electrodes] -> tokens [B, (T/patch)*n_electrodes, dim]."""

    def __init__(self, config, verbose: bool = False):
        super().__init__()
        self.config = config
        self.patch_size = config.patch_size
        self.n_electrodes = config.n_electrodes
        self.n_patches_per_channel = config.window_size // config.patch_size
        self.block_size = self.n_patches_per_channel * config.n_electrodes
        self.transformer = nn.ModuleDict(dict(
            emb=nn.Linear(config.patch_size, config.dim),
            h=nn.ModuleList([Block(config) for _ in range(config.n_layers)]),
            ln_f=_KernelLayerNorm(config.dim),
        ))
        self.space_embedding = nn.Parameter(torch.randn(1, config.n_electrodes, config.dim), requires_grad=True)
        self.precompute_rope_cash = build_complex_rope_cache(dim=config.head_dim, seq_len=self.block_size,
                                                             theta=config.rope_theta)
        # kept only so that checkpoints written by the reference load with strict=True; never read by a kernel
        self.register_buffer('attn_mask', build_advanced_causal_mask(self.block_size, self.n_electrodes))
        self._rope_table = None
        if verbose:
            print("Encoder: number of parameters: %.2fM" % (self.get_num_params() / 1e6,))

    def to_patches(self, x):
        """'b (t p1) c -> b (t c) p1': token = (time patch, electrode), electrode fastest (brainformer.py:282)."""
        b, T, c = x.shape
        p = self.patch_size
        if T % p != 0:
            raise ValueError(f"window of {T} bins is not divisible by patch_size {p}")
        return x.view(b, T // p, p, c).transpose(2, 3).reshape(b, (T // p) * c, p)

    @property
    def dtype(self) -> torch.dtype:
        return next(self.parameters()).dtype

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    @property
    def rope_cache(self) -> torch.Tensor:
        if self.precompute_rope_cash.device != self.device:
            self.precompute_rope_cash = self.precompute_rope_cash.to(device=self.device)
        return self.precompute_rope_cash

    def rope_table(self) -> torch.Tensor:
        """fp32 [block_size, head_dim/2, 2] view of the complex cache for the RoPE kernel."""
        if self._rope_table is None or self._rope_table.device != self.device:
            self._rope_table = torch.view_as_real(self.rope_cache).float().contiguous()
        return self._rope_table

    @property
    def spatial_pos_embedding(self):
        return self.space_embedding.repeat((1, self.n_patches_per_channel, 1))

    def get_num_params(self):
        return sum(p.numel() for p in self.parameters())

    def embed(self, patches):
        return _linear_bf16(patches, self.transformer.emb.weight, self.transformer.emb.bias)

    def forward(self, x, kv_cache=None, out_dtype=torch.float32):
        """out_dtype: dtype of the final LayerNorm output (the perceiver asks for bf16, the operand type of its GEMMs)."""
        b, T, E = x.shape
        if T % self.patch_size != 0:
            raise ValueError(f"window of {T} bins is not divisible by patch_size {self.patch_size}")
        n_tokens = (T // self.patch_size) * E
        w_emb = self.transformer.emb
        fused = (GEMM_IMPL == "own" and x.is_cuda and not x.requires_grad
                 and gemm.patch_embed_supported(T, E, self.patch_size, w_emb.weight.shape[0]))
        if fused:
            # patchify + Linear(p -> dim) + bias as ONE tcgen05 contraction fed by TMA straight from x (csrc/gemm.cu,
            # fk_patch_embed_forward): the [B, S, p] patch tensor of `to_patches` is never written
            h_delta = gemm.patch_embed(x, w_emb.weight, w_emb.bias)
        else:
            h_delta = self.embed(self.to_patches(x))
        emb = self.spatial_pos_embedding[:, -n_tokens:].float()       # [1, S, dim]; added inside the first add+LayerNorm
        mask = LabelMask.block_causal(b, n_tokens, self.n_electrodes, x.device)
        if n_tokens != self.block_size:
            # the reference slices attn_mask[-T:, -T:] and rope[-T:]: labels of the LAST n_tokens positions
            first = self.block_size - n_tokens
            ids = ((torch.arange(n_tokens, device=x.device) + first) // self.n_electrodes).to(torch.int32)
            mask = LabelMask(ids[None].expand(b, n_tokens).contiguous())
        rope = RopeSpec(self.rope_table(), None, self.block_size - n_tokens)
        _, y = run_blocks(self.transformer.h, emb, mask, rope, self.transformer.ln_f, out_dtype, h_delta=h_delta)
        return y

    def stream(self, batch_size: int, out_dtype=torch.float32, sliding: bool = False) -> "EncoderStream":
        """Online inference: feed the window patch by patch with `EncoderStream.step(x)` and get the outputs of the new
        tokens only.  The mask is block-causal per time patch, so earlier tokens' outputs never change; each layer keeps the
        rotated keys and values of the tokens seen so far in a bf16 cache of `block_size` tokens.

        sliding=True: a stream with no end.  A token at every layer attends to the tokens of its own time patch and of the
        W - 1 patches before it (W = window_size // patch_size, the model's window), so within the first window this is the
        model exactly and past it every query sees the relative distances the model was trained on.  Each layer keeps a
        ring cache of 2 W patches instead of the window."""
        return EncoderStream(self, batch_size, out_dtype, sliding)


class EncoderStream:
    """Streaming state of an `Encoder` (from `Encoder.stream`): per layer a bf16 k | v cache [B, block_size, 2 * inner],
    allocated once.  Positions start at 0 when the stream starts; the offline `Encoder.forward` on a partial window uses
    the last positions of the window instead, a uniform shift that RoPE scores do not see, so the two agree up to bf16
    rounding.

    Each batch row is a session of its own: `reset(rows)` restarts only the given rows, and from then on the rows sit at
    different positions (`lengths`).  A step advances every row by the same whole patches, or, with `counts`, each row by
    its own count (0 included: a session with no new data waits); each row continues at its own position, and its outputs
    depend on its own session only.  Until the first per-row reset or step with differing counts (and again after
    `reset()`) every row is at one position and a step runs the lockstep path.

    The caches hold one scratch row past the last row's window: the k | v rows of the slots past a row's count go there,
    so no filler ever enters a window.

    Sliding (`Encoder.stream(..., sliding=True)`): no length limit.  Each layer's cache is a ring of 2 W patches per row
    (W patches in the band of the newest query plus up to W new ones), token p in slot p mod 2 W E, and the attention
    takes a label band of W patches (ops.LabelMask band) over the whole ring.  The ring slots' key labels (p // E, INT_MAX
    for a slot no session of the row has written) and the RoPE rows of the new positions, computed in fp64, come from one
    launch per step (fk_stream_ring_positions).  Every step takes the per-row path; a step gives a row at most W patches."""

    def __init__(self, encoder: Encoder, batch_size: int, out_dtype=torch.float32, sliding: bool = False):
        cfg = encoder.config
        if batch_size < 1:
            raise ops.FkError("EncoderStream: batch_size must be positive")
        if cfg.head_dim not in (16, 32, 64):
            raise ops.FkError("EncoderStream: the streaming attention kernel takes head_dim 16, 32 or 64")
        if len(encoder.transformer.h) == 0:
            raise ops.FkError("EncoderStream: the encoder has no layers")
        self.encoder = encoder
        self.batch_size = batch_size
        self.out_dtype = out_dtype
        self.sliding = bool(sliding)
        self.n_heads = cfg.n_heads
        self.inner = cfg.n_heads * cfg.head_dim
        self.window = encoder.n_patches_per_channel                       # W patches: the band of a sliding stream
        self.cap = 2 * encoder.block_size if self.sliding else encoder.block_size   # cache tokens per row
        dev = encoder.device
        # zeroed: a row's partly visible key tile multiplies P = 0 by the V rows past its length (fk_attn_forward_kv_tc).
        # Flat [B * cap + 1, 2 * inner]: the last row takes the k | v rows of slots past a row's count.
        self._flat = [torch.zeros(batch_size * self.cap + 1, 2 * self.inner, device=dev, dtype=BF16)
                      for _ in encoder.transformer.h]
        self.caches = [f[:-1].view(batch_size, self.cap, 2 * self.inner) for f in self._flat]
        self._lengths = [0] * batch_size
        # per-row sessions: device lengths in two buffers (a step reads one and writes the other, the roles swap once the
        # step is enqueued) and the key labels of the whole window, shared by every row and built on first use
        self._ragged = self.sliding
        self._len_dev = torch.zeros(2, batch_size, device=dev, dtype=torch.int64 if self.sliding else torch.int32)
        self._cur = 0
        self._keys = None
        if self.sliding:
            # ring key labels [B, cap] with their 64-slot tile ranges, INT_MAX (seen by no query) until a session writes
            # the slot; the ring kernel keeps them current
            nt = (self.cap + 63) // 64
            kid = torch.full((batch_size, self.cap), _INT32_MAX, device=dev, dtype=torch.int32)
            kmin = torch.full((batch_size, nt), _INT32_MAX, device=dev, dtype=torch.int32)
            self._keys = LabelMask.from_ranges(None, kid, None, None, kmin, kmin.clone())
            self._inv_freq = rope_inv_freq(cfg.head_dim, cfg.rope_theta).to(dev)
            self._rope_pos = {}

    @property
    def lengths(self) -> list:
        """tokens cached so far, per row (host values: reading them does not wait for the device)."""
        return list(self._lengths)

    @property
    def length(self) -> int:
        """tokens cached so far (a multiple of n_electrodes), while every row is at the same position."""
        return ops.stream_length(self._lengths, "EncoderStream.length")

    def reset(self, rows=None) -> None:
        """Restart every row (rows None) or only the given row indices; FkError, changing nothing, for an index outside
        the batch or a duplicate."""
        if rows is None:
            self._lengths = [0] * self.batch_size
            self._ragged = self.sliding
            if self.sliding:
                self._len_dev[self._cur].zero_()
                for t in (self._keys.kid, self._keys.kmin, self._keys.kmax):
                    t.fill_(_INT32_MAX)
            return
        idx = ops.stream_rows(rows, self.batch_size, "EncoderStream.reset")
        if not idx:
            return
        cur = self._to_ragged()
        sel = torch.tensor(idx, dtype=torch.long).to(cur.device)
        cur.index_fill_(0, sel, 0)
        if self.sliding:
            # the ring slots of the rows' earlier sessions: a restarted session must not see them once its own patch
            # index passes their labels
            for t in (self._keys.kid, self._keys.kmin, self._keys.kmax):
                t.index_fill_(0, sel, _INT32_MAX)
        for r in idx:
            self._lengths[r] = 0

    def _to_ragged(self):
        """the current device lengths, filled from the host on leaving the lockstep path (which keeps them on the host only)"""
        cur = self._len_dev[self._cur]
        if not self._ragged:
            cur.fill_(self._lengths[0])
            self._ragged = True
        return cur

    def _key_labels(self):
        """block-causal labels of every cache position, [B, block_size], with their tile ranges (built once)."""
        if self._keys is None:
            enc = self.encoder
            kid = torch.arange(enc.block_size, device=self._len_dev.device, dtype=torch.int32) // enc.n_electrodes
            self._keys = LabelMask(kid[None].expand(self.batch_size, -1).contiguous())
        return self._keys

    @torch.no_grad()
    def step(self, x: torch.Tensor, counts=None) -> torch.Tensor:
        """x [B, n * patch_size, n_electrodes] (n >= 1 whole patches) -> final-LayerNorm outputs of the n * n_electrodes
        new tokens, [B, n * n_electrodes, dim] in `out_dtype`.

        counts: optional host sequence of B ints, the whole patches of x that are new data for each row (0 ... n).  Row b
        advances by counts[b] patches; the rest of its bins are ignored whatever they hold (NaN included), and its token
        slots past counts[b] * n_electrodes are zero.  None, or every count n, is the plain step.

        Raises FkError, leaving the state as it was, on a partial patch, a batch or electrode count that does not match, bad
        counts (number, range), or a step that takes any row past the window (block_size tokens).  A sliding stream has no
        window limit; it raises instead for a step that gives a row more than W patches or takes its patch index past int32."""
        return self._step(x, counts)[0]

    def _step(self, x, counts=None):
        """step(x, counts) and, for rows at different positions, the flat cache rows b * block_size + position that the new
        tokens took, B * block_size for slots past a row's count (int64 [B * n_new]; None on the lockstep path)."""
        enc = self.encoder
        E, p = enc.n_electrodes, enc.patch_size
        if x.dim() != 3 or x.shape[0] != self.batch_size or x.shape[2] != E:
            raise ops.FkError(f"EncoderStream.step: expected [{self.batch_size}, n * {p}, {E}], got {tuple(x.shape)}")
        B, T, _ = x.shape
        if T < p or T % p != 0:
            raise ops.FkError(f"EncoderStream.step: {T} bins is not a positive multiple of patch_size {p}")
        n_new = (T // p) * E
        if counts is not None:
            counts = ops.stream_counts(counts, B, T // p, 1, "EncoderStream.step")
            if all(c == T // p for c in counts):
                counts = None                          # every row takes the whole step: the plain step
        adv = [n_new] * B if counts is None else [c * E for c in counts]
        if self.sliding:
            return self._step_sliding(x, counts, adv)
        over = [b for b, n in enumerate(self._lengths) if n + adv[b] > enc.block_size]
        if over:
            raise ops.FkError(f"EncoderStream.step: {[adv[b] for b in over]} new tokens take rows {over} (at "
                              f"{[self._lengths[b] for b in over]} tokens) past the window of {enc.block_size}")
        if not x.is_cuda:
            raise ops.FkError("frankenstein_b200 modules run on a B200 only (no CPU fallback)")
        cnt = None
        if counts is not None:
            self._to_ragged()
            cnt = torch.tensor(adv, dtype=torch.int32).to(x.device)     # the one host-to-device copy of the step
        w_emb = enc.transformer.emb
        if GEMM_IMPL == "own" and gemm.patch_embed_supported(T, E, p, w_emb.weight.shape[0]):
            h_delta = gemm.patch_embed(x.detach(), w_emb.weight, w_emb.bias)
        else:
            h_delta = enc.embed(enc.to_patches(x))
        emb = enc.space_embedding.float().repeat(1, T // p, 1)        # [1, n_new, dim]; added inside the first add+LayerNorm
        rows = None
        if not self._ragged:
            L = self._lengths[0]
            Sk = L + n_new
            mask = None
            if T > p:
                # several patches in one step: block-causal among the new tokens (with one patch every cached key is visible)
                blk = torch.arange(Sk, device=x.device, dtype=torch.int32) // E
                mask = LabelMask(blk[L:][None].expand(B, n_new).contiguous(), blk[None].expand(B, Sk).contiguous())
            rope = RopeSpec(enc.rope_table(), None, L)
        else:
            # rows at different positions: one launch gives each row's query labels, RoPE positions and cache rows.  The
            # attention runs over the whole window with fixed key labels, so its key chunks do not depend on the other
            # rows' lengths; cached positions at or past a row's length belong to later time patches and are masked
            # (whole tiles of them are skipped by the tile ranges).
            keys = self._key_labels()
            # With counts, the slots past a row's count see no key and write their k | v to the scratch row.
            qid, qmin, qmax, pos, rows = ops.stream_positions(self._len_dev[self._cur], self._len_dev[self._cur ^ 1], n_new, E,
                                                              enc.block_size, cnt)
            mask = LabelMask.from_ranges(qid, keys.qid, qmin, qmax, keys.qmin, keys.qmax)
            rope = RopeSpec(enc.rope_table(), pos, 0)
            Sk = enc.block_size
        blocks = enc.transformer.h
        H, inner = self.n_heads, self.inner
        l0 = blocks[0].ln_1
        h, y = ops.add_layer_norm(emb, h_delta, l0.weight, l0.bias, l0.eps)
        for i, blk_ in enumerate(blocks):
            at = blk_.attn
            if GEMM_IMPL == "own" and gemm.qkv_supported(at.qw.weight.shape[1], inner):
                qkv = gemm.qkv_rope(y, at.qw.weight, at.kw.weight, at.vw.weight, rope, H)
            else:
                qkv = _linear_bf16(y, torch.cat([at.qw.weight, at.kw.weight, at.vw.weight], dim=0)).contiguous()
                q4 = qkv.view(B, n_new, 3, H, -1)
                ops._rope_inplace(q4[:, :, 0], rope, False)
                ops._rope_inplace(q4[:, :, 1], rope, False)
            cache = self.caches[i]
            if rows is None:
                cache[:, L:Sk].copy_(qkv[..., inner:])
            else:
                self._flat[i].index_copy_(0, rows, qkv[..., inner:].reshape(-1, 2 * inner))
            res = ops.attention_kv(qkv[..., :inner], cache[:, :Sk, :inner], cache[:, :Sk, inner:], H, mask)
            a = _linear_bf16(res, at.project.weight)
            h, y = ops.add_layer_norm(h, a, blk_.ln_2.weight, blk_.ln_2.bias, blk_.ln_2.eps)
            m = blk_.mlp(y)
            nxt = blocks[i + 1].ln_1 if i + 1 < len(blocks) else enc.transformer.ln_f
            h, y = ops.add_layer_norm(h, m, nxt.weight, nxt.bias, nxt.eps,
                                      BF16 if i + 1 < len(blocks) else self.out_dtype)
        if cnt is not None:
            y.masked_fill_((qid == ops.NO_LABEL)[..., None], 0)      # token slots past each row's count
        if self._ragged:
            self._cur ^= 1
        self._lengths = [n + a for n, a in zip(self._lengths, adv)]
        return y, rows

    def _step_sliding(self, x, counts, adv):
        """_step of a sliding stream: the ring bookkeeping in one launch, each layer's new k | v rows into its ring, and the
        banded attention over the whole ring (a fixed key axis, so a row's bits depend on its own session only)."""
        enc = self.encoder
        E, p, W = enc.n_electrodes, enc.patch_size, self.window
        B, T, _ = x.shape
        n_new = (T // p) * E
        over = [b for b in range(B) if adv[b] > W * E]
        if over:
            raise ops.FkError(f"EncoderStream.step: rows {over} get {[adv[b] // E for b in over]} patches in one step; a "
                              f"sliding stream takes at most W = {W} per row and step")
        over = [b for b in range(B) if adv[b] and (self._lengths[b] + adv[b] - 1) // E > _INT32_MAX]
        if over:
            raise ops.FkError(f"EncoderStream.step: rows {over} (at {[self._lengths[b] for b in over]} tokens) would take "
                              "their patch index past int32; reset them")
        if not x.is_cuda:
            raise ops.FkError("frankenstein_b200 modules run on a B200 only (no CPU fallback)")
        cnt = None if counts is None else torch.tensor(adv, dtype=torch.int32).to(x.device)   # the step's host-to-device copy
        w_emb = enc.transformer.emb
        if GEMM_IMPL == "own" and gemm.patch_embed_supported(T, E, p, w_emb.weight.shape[0]):
            h_delta = gemm.patch_embed(x.detach(), w_emb.weight, w_emb.bias)
        else:
            h_delta = enc.embed(enc.to_patches(x))
        emb = enc.space_embedding.float().repeat(1, T // p, 1)
        keys = self._keys
        qid, qmin, qmax, rows, table = ops.stream_ring_positions(self._len_dev[self._cur], self._len_dev[self._cur ^ 1], n_new,
                                                                 E, self.cap, keys, self._inv_freq, cnt)
        mask = LabelMask.from_ranges(qid, keys.kid, qmin, qmax, keys.kmin, keys.kmax, band=W)
        if n_new not in self._rope_pos:
            self._rope_pos[n_new] = torch.arange(B * n_new, device=x.device, dtype=torch.int32).view(B, n_new)
        rope = RopeSpec(table, self._rope_pos[n_new], 0)               # row b * n_new + i of this step's table
        blocks = enc.transformer.h
        H, inner = self.n_heads, self.inner
        l0 = blocks[0].ln_1
        h, y = ops.add_layer_norm(emb, h_delta, l0.weight, l0.bias, l0.eps)
        for i, blk_ in enumerate(blocks):
            at = blk_.attn
            if GEMM_IMPL == "own" and gemm.qkv_supported(at.qw.weight.shape[1], inner):
                qkv = gemm.qkv_rope(y, at.qw.weight, at.kw.weight, at.vw.weight, rope, H)
            else:
                qkv = _linear_bf16(y, torch.cat([at.qw.weight, at.kw.weight, at.vw.weight], dim=0)).contiguous()
                q4 = qkv.view(B, n_new, 3, H, -1)
                ops._rope_inplace(q4[:, :, 0], rope, False)
                ops._rope_inplace(q4[:, :, 1], rope, False)
            cache = self.caches[i]
            self._flat[i].index_copy_(0, rows, qkv[..., inner:].reshape(-1, 2 * inner))
            res = ops.attention_kv(qkv[..., :inner], cache[..., :inner], cache[..., inner:], H, mask)
            a = _linear_bf16(res, at.project.weight)
            h, y = ops.add_layer_norm(h, a, blk_.ln_2.weight, blk_.ln_2.bias, blk_.ln_2.eps)
            m = blk_.mlp(y)
            nxt = blocks[i + 1].ln_1 if i + 1 < len(blocks) else enc.transformer.ln_f
            h, y = ops.add_layer_norm(h, m, nxt.weight, nxt.bias, nxt.eps,
                                      BF16 if i + 1 < len(blocks) else self.out_dtype)
        if cnt is not None:
            y.masked_fill_((qid == ops.NO_LABEL)[..., None], 0)      # token slots past each row's count
        self._cur ^= 1
        self._lengths = [n + a for n, a in zip(self._lengths, adv)]
        return y, rows


class MAE(nn.Module):
    """Masked auto-encoder pre-training  (models/brainformer.py:354-486)."""

    def __init__(self, config, verbose: bool = False):
        super().__init__()
        self.config = config
        self.decoder_dim = config.decoder_dim
        self.encoder = Encoder(config, verbose)
        self.decoder = nn.ModuleDict(dict(
            emb=nn.Identity(),
            h=nn.ModuleList([Block(config) for _ in range(config.n_dec_layers)]),
        ))
        self.mask_token = nn.Parameter(torch.randn(config.dim))
        self.decoder_pos_emb = nn.Embedding(self.encoder.block_size, config.decoder_dim)
        self.to_signals = nn.Linear(config.decoder_dim, config.patch_size)
        if verbose:
            print("MAE: number of parameters: %.2fM" % (self.get_num_params() / 1e6))

    def get_num_params(self, non_embedding=True):
        return sum(p.numel() for p in self.parameters())

    def to_signal_shape(self, tokens):
        """'b (t c) p -> b (t p) c' (brainformer.py:371)."""
        b, n, p = tokens.shape
        c = self.config.n_electrodes
        return tokens.view(b, n // c, c, p).transpose(2, 3).reshape(b, (n // c) * p, c)

    def get_masking_indices(self, masking_ratio, x):
        """uniform scores -> argsort -> split -> sort each part (brainformer.py:380-390)."""
        b, n_tokens, _ = x.shape
        num_masked = int(masking_ratio * n_tokens)
        order = torch.rand(b, n_tokens, device=x.device).argsort(dim=-1)
        masked, unmasked = order[:, :num_masked], order[:, num_masked:]
        return torch.sort(masked, dim=1)[0], torch.sort(unmasked, dim=1)[0]

    def get_sub_att_matrix(self, attn_mask, unmasked_indices):
        """dense [b,1,s,s] sub-mask as in brainformer.py:392-413 (API compatibility; forward() uses labels)."""
        sub = attn_mask[unmasked_indices[:, :, None], unmasked_indices[:, None, :]]
        return sub[:, None]

    def forward(self, x, targets=None, date_info=None, masking_ratio=0.75, return_preds=False):
        enc = self.encoder
        x = enc.to_patches(x)
        b, n_tokens, _ = x.shape
        masked_indices, unmasked_indices = self.get_masking_indices(masking_ratio, x)
        rows = torch.arange(b, device=x.device)[:, None]

        # ---- encoder on the kept tokens: per-sample electrode embedding, rope position and mask labels ----
        kept = x[rows, unmasked_indices]
        tokens = enc.embed(kept) + enc.spatial_pos_embedding[0][unmasked_indices]
        mask = LabelMask((unmasked_indices // enc.n_electrodes).to(torch.int32))
        rope = RopeSpec(enc.rope_table(), unmasked_indices, 0)
        _, tokens = run_blocks(enc.transformer.h, tokens, mask, rope, enc.transformer.ln_f)

        # ---- decoder on all tokens (no mask, no rope); pos-emb order is cat[unmasked, masked] as in the reference ----
        dec = torch.zeros(b, n_tokens, self.decoder_dim, device=x.device, dtype=tokens.dtype)
        dec[rows, unmasked_indices] = self.decoder.emb(tokens)
        dec[rows, masked_indices] = self.mask_token.to(dec.dtype)
        dec = dec + self.decoder_pos_emb(torch.cat([unmasked_indices, masked_indices], 1))
        dec, _ = run_blocks(self.decoder.h, dec)

        pred = _linear_bf16(dec[rows, masked_indices], self.to_signals.weight, self.to_signals.bias).float()
        target = x[rows, masked_indices]
        recon_loss = F.mse_loss(pred, target)
        if return_preds:
            binary_mask = torch.zeros_like(x)
            binary_mask[rows, masked_indices] = 1
            recon = torch.zeros_like(x)
            recon[rows, masked_indices] = pred.to(x.dtype)
            recon[rows, unmasked_indices] = kept
            return recon_loss, self.to_signal_shape(recon), self.to_signal_shape(binary_mask)
        return (recon_loss, None)


class BrainFormer(nn.Module):
    """Encoder + perceiver resampler  (models/brainformer.py:488-574)."""
    config = Config

    def __init__(self, config: Config, verbose: bool = False):
        super().__init__()
        self.config = config
        self.encoder = Encoder(config.encoder, verbose)
        self.n_output_tokens = config.n_output_tokens
        self.learnable_queries = nn.Parameter(torch.zeros(1, config.n_output_tokens, config.dim))
        self.perceiver = nn.ModuleDict(dict(
            h=nn.ModuleList([CrossBlock(config) for _ in range(config.n_layers)]),
            ln_f=_KernelLayerNorm(config.dim),
            to_motion=nn.Linear(config.dim, config.output_dim)))
        self.register_buffer('cross_attn_mask', None)
        self.register_buffer('self_attn_mask', None)
        self.precompute_rope_cash = build_complex_rope_cache(dim=config.head_dim, seq_len=config.n_output_tokens,
                                                             theta=config.rope_theta)
        if verbose:
            print("Full HandFormer: number of parameters: %.2fM" % (self.get_num_params() / 1e6,))

    def get_num_params(self):
        return sum(p.numel() for p in self.parameters())

    @property
    def dtype(self) -> torch.dtype:
        return next(self.parameters()).dtype

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    @property
    def rope_cache(self) -> torch.Tensor:
        if self.precompute_rope_cash.device != self.device:
            self.precompute_rope_cash = self.precompute_rope_cash.to(device=self.device)
        return self.precompute_rope_cash

    def forward(self, x, targets=None, date_info=None):
        b = x.shape[0]
        context = self.encoder(x, out_dtype=BF16)
        h = self.learnable_queries.expand(b, self.n_output_tokens, -1)
        for cross_block in self.perceiver.h:
            h = cross_block(h, context, self.self_attn_mask, self.cross_attn_mask, sa_rope=self.rope_cache)
        pred = self.perceiver.ln_f(h)
        pred = _linear_bf16(pred, self.perceiver.to_motion.weight, self.perceiver.to_motion.bias).float()
        if targets is None:
            return None, pred
        return F.l1_loss(pred, targets), pred

    @torch.no_grad()
    def inference(self, myo, date_info):
        x = torch.from_numpy(myo)[None].to(self.device).to(self.dtype)
        return self.forward(x, targets=None)[1][0].detach().cpu().numpy().T

    def stream(self, batch_size: int, sliding: bool = False) -> "BrainFormerStream":
        """Online decoding: `BrainFormerStream.step(x)` takes the next whole patches of the window and returns `pred` as
        `forward` would for every bin fed so far.  sliding=True: a stream with no end (see `Encoder.stream`); `pred` is the
        perceiver over the context tokens of the last W patches."""
        return BrainFormerStream(self, batch_size, sliding)


class BrainFormerStream:
    """Streaming state of a `BrainFormer`: an `EncoderStream` plus, per CrossBlock, a bf16 cache of the k | v projection
    of the context tokens [B, block_size, 2 * inner].  The encoder is block-causal, so the context tokens never change
    once produced: a step projects only the new ones, then runs the perceiver over the whole cache in place.  Batch rows
    are sessions of their own as in `EncoderStream`: after `reset(rows)`, or in a step with per-row `counts`, the perceiver
    of each row reads that row's own context tokens only.  Like the encoder's caches, each context cache holds one scratch
    row past the last row's window for the slots past a row's count.

    Sliding (`BrainFormer.stream(..., sliding=True)`): each context cache is a ring of exactly W patches (block_size
    tokens) per row, token p in slot p mod block_size, so the valid slots are a prefix until the ring wraps and all of it
    afterwards.  Cross-attention has no mask and no RoPE, so slot order does not matter: the perceiver reads the first
    min(length, block_size) slots of each row, the context tokens of its last W patches."""

    def __init__(self, model: BrainFormer, batch_size: int, sliding: bool = False):
        cfg = model.config
        if not ops.small_attention_supported(model.n_output_tokens, cfg.head_dim):
            raise ops.FkError("BrainFormerStream: the cross-attention kernel serves <= 64 queries at head_dim 16 / 32 / 64")
        self.model = model
        self.encoder_stream = model.encoder.stream(batch_size, out_dtype=BF16, sliding=sliding)
        inner = cfg.n_heads * cfg.head_dim
        block = model.encoder.block_size
        self._flat = [torch.zeros(batch_size * block + 1, 2 * inner, device=model.device, dtype=BF16) for _ in model.perceiver.h]
        self.kv = [f[:-1].view(batch_size, block, 2 * inner) for f in self._flat]

    @property
    def lengths(self) -> list:
        """context tokens cached so far, per row."""
        return self.encoder_stream.lengths

    @property
    def length(self) -> int:
        """context tokens cached so far, while every row is at the same position."""
        return self.encoder_stream.length

    def reset(self, rows=None) -> None:
        """Restart every row (rows None) or only the given row indices (see `EncoderStream.reset`)."""
        self.encoder_stream.reset(rows)

    @torch.no_grad()
    def step(self, x: torch.Tensor, counts=None) -> torch.Tensor:
        """x [B, n * patch_size, n_electrodes] -> pred [B, n_output_tokens, output_dim] fp32 over every row's context so far
        (errors as EncoderStream.step).  counts: optional per-row whole patches of new data, as in `EncoderStream.step`; a
        row with count 0 gets its prediction again, and a row with no context yet the perceiver over an empty context."""
        m = self.model
        es = self.encoder_stream
        L0 = es.lengths[0]
        context, rows = es._step(x, counts)                        # [B, n_new, dim] bf16
        L = max(es.lengths)
        k_len = None if rows is None else es._len_dev[es._cur]     # the rows' lengths after this step
        if es.sliding:
            # ring row b * C + p mod C of the encoder ring row b * 2C + p mod 2C (the scratch row B * 2C -> B * C)
            C = m.encoder.block_size
            rows = rows // es.cap * C + rows % C
            k_len = k_len.clamp(max=C).to(torch.int32)
            L = C
        for cb, kv, flat in zip(m.perceiver.h, self.kv, self._flat):
            ca = cb.cross_attn
            proj = _linear_bf16(context, torch.cat([ca.kw.weight, ca.vw.weight], dim=0))
            if rows is None:
                kv[:, L0:L].copy_(proj)
            else:
                flat.index_copy_(0, rows, proj.reshape(-1, kv.shape[-1]))
        h = m.learnable_queries.expand(x.shape[0], m.n_output_tokens, -1)
        for cb, kv in zip(m.perceiver.h, self.kv):
            ca = cb.cross_attn
            q = _linear_bf16(cb.ln_1(h), ca.qw.weight)
            res = ops.small_attention_kv_cached(q, kv[:, :max(L, 1)], ca.n_heads, k_len=k_len)   # k_len 0: a zero row
            h = h + _linear_bf16(res, ca.project.weight)
            h = h + cb.mlp(cb.ln_2(h))
            h = cb.sa_block(h, attn_mask=m.self_attn_mask, rope=m.rope_cache)
        pred = m.perceiver.ln_f(h)
        return _linear_bf16(pred, m.perceiver.to_motion.weight, m.perceiver.to_motion.bias).float()
