"""torch.autograd wrappers over the transformer-block kernels of libfk_b200.so.

LayerNorm / RMSNorm, SwiGLU gate, RoPE and masked flash attention, each a thin
``torch.autograd.Function`` that passes raw device pointers + the current stream through the C ABI
(include/fk_b200.h).  CPU tensors raise: there is no fallback path.
"""
from __future__ import annotations

import operator
from typing import Optional

import torch

from . import _lib
from ._lib import FkError, check, counters, lib, on_tensor_device, ptr, require_cuda, require_device, stream, timed

_DT = {torch.float32: 0, torch.bfloat16: 1}

import os

COLSUM_IMPL = os.environ.get("FK_COLSUM", "own")        # bias gradients: "own" = fk_colsum_partials, "torch" = g.sum(0, dtype=float32)
# attention backward implementation: "tc" = tcgen05/TMEM/TMA kernels (attention_tc.cu), "legacy" = mma.sync kernels
ATTN_BWD_IMPL = os.environ.get("FK_ATTN_BWD", "tc")
ATTN_FWD_IMPL = os.environ.get("FK_ATTN_FWD", "tc")
# B operand of the backward accumulate MMAs: "mn" = MN-major straight from the [tokens][32] tiles (no copies),
# "transposed" = K-major from token-contiguous copies made by fk_attn_transpose (cross-check path)
ATTN_BWD_OPERANDS = os.environ.get("FK_ATTN_BWD_OPERANDS", "mn")
# row statistics of the backward: "folded" = -lse / c and -delta enter the score MMAs as one more K step (fk_attn_aug),
# "staged" = read from lse / delta and subtracted by the compute warps (cross-check path)
ATTN_BWD_STATS = os.environ.get("FK_ATTN_BWD_STATS", "folded")


# ------------------------------------------------------------------------------------------------
# LayerNorm / RMSNorm
# ------------------------------------------------------------------------------------------------
def _reduce_partials(dwp, dbp, w_dtype):
    """dweight / dbias from the per-block partial sums of the norm backward: one launch for both, fixed order."""
    nb, D = dwp.shape
    dw = torch.empty(D, device=dwp.device, dtype=torch.float32)
    db = torch.empty(D, device=dwp.device, dtype=torch.float32) if dbp is not None else None
    check(lib().fk_norm_reduce_partials(ptr(dwp), ptr(dbp), nb, D, ptr(dw), ptr(db), stream()), "fk_norm_reduce_partials")
    return dw.to(w_dtype), (db.to(w_dtype) if db is not None else None)


def column_sum(g2: torch.Tensor) -> torch.Tensor:
    """fp32 column sums of a bf16 [M, N] matrix (bias gradient of a Linear / Conv1d: sum of dY over the tokens), two launches,
    fixed summation order.  Falls back to torch's reduction for layouts the kernel does not take."""
    M, N = g2.shape
    if (COLSUM_IMPL != "own" or g2.dtype != torch.bfloat16 or N % 8 != 0 or g2.stride(1) != 1 or g2.stride(0) % 8 != 0
            or g2.stride(0) < N or g2.data_ptr() % 16 != 0 or M * N < (1 << 23) or g2.device.index != torch.cuda.current_device()):
        return g2.sum(0, dtype=torch.float32)          # (below ~8 M elements one torch launch beats two of ours: launch-bound)
    nb = lib().fk_colsum_grid()
    part = torch.empty(nb, N, device=g2.device, dtype=torch.float32)
    out = torch.empty(N, device=g2.device, dtype=torch.float32)
    check(lib().fk_colsum_partials(ptr(g2), M, N, g2.stride(0), ptr(part), stream()), "fk_colsum_partials")
    check(lib().fk_norm_reduce_partials(ptr(part), None, nb, N, ptr(out), None, stream()), "fk_norm_reduce_partials")
    return out


class _NormFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, x, weight, bias, eps, rms, out_dtype):
        require_cuda(x, weight)
        require_device()
        D = x.shape[-1]
        xc = x.contiguous()
        if xc.dtype not in _DT or (xc.dtype == torch.bfloat16 and out_dtype == torch.float32):
            xc = xc.float()
        M = xc.numel() // D
        w = weight.detach().float().contiguous()
        b = bias.detach().float().contiguous() if bias is not None else None
        y = torch.empty(x.shape, device=x.device, dtype=out_dtype)
        mean = None if rms else torch.empty(M, device=x.device, dtype=torch.float32)
        rstd = torch.empty(M, device=x.device, dtype=torch.float32)
        check(lib().fk_norm_forward(ptr(xc), _DT[xc.dtype], ptr(w), ptr(b), ptr(y), _DT[out_dtype], ptr(mean), ptr(rstd),
                                    M, D, float(eps), int(rms), stream()), "fk_norm_forward")
        ctx.save_for_backward(xc, w, mean if mean is not None else torch.empty(0, device=x.device), rstd)
        ctx.rms = rms
        ctx.has_bias = bias is not None
        ctx.in_dtype = x.dtype
        ctx.w_dtype = weight.dtype
        return y

    @staticmethod
    @on_tensor_device
    def backward(ctx, g):
        xc, w, mean, rstd = ctx.saved_tensors
        D = xc.shape[-1]
        M = xc.numel() // D
        g = g.contiguous()
        # supported (x, g, dx) combinations of the kernel
        if xc.dtype == torch.float32 and g.dtype not in _DT:
            g = g.float()
        if xc.dtype == torch.bfloat16 and g.dtype != torch.bfloat16:
            g = g.to(torch.bfloat16)
        dx = torch.empty_like(xc)
        nb = lib().fk_norm_backward_grid()
        dwp = torch.empty(nb, D, device=xc.device, dtype=torch.float32)
        dbp = torch.empty(nb, D, device=xc.device, dtype=torch.float32) if ctx.has_bias else None
        check(lib().fk_norm_backward(ptr(xc), _DT[xc.dtype], ptr(g), _DT[g.dtype], ptr(w), ptr(mean) if not ctx.rms else 0,
                                     ptr(rstd), ptr(dx), _DT[dx.dtype], ptr(dwp), ptr(dbp), M, D, int(ctx.rms), stream()),
              "fk_norm_backward")
        dw, db = _reduce_partials(dwp, dbp, ctx.w_dtype)
        return dx.to(ctx.in_dtype), dw, db, None, None, None


class _AddNormFn(torch.autograd.Function):
    """(x_new, y) = (x + delta, norm(x + delta)) in one pass over the fp32 residual stream; backward fuses the norm
    backward with the residual-gradient add and emits the bf16 gradient of the delta branch."""

    @staticmethod
    @on_tensor_device
    def forward(ctx, x, delta, weight, bias, eps, rms, out_dtype):
        require_cuda(x, delta, weight)
        require_device()
        if x.dtype != torch.float32 or delta.dtype != torch.bfloat16:
            raise FkError("add_norm expects an fp32 residual stream and a bf16 branch output")
        D = x.shape[-1]
        xc, dc = x.contiguous(), delta.contiguous()
        M = dc.numel() // D
        period = 0
        if xc.numel() != dc.numel():
            # x [1, S, D] broadcast over the batch of delta [B, S, D] (embedding table + patch projection)
            if xc.dim() != dc.dim() or xc.shape[0] != 1 or xc.shape[1:] != dc.shape[1:]:
                raise FkError("add_norm: x must match delta or be [1, ...] broadcast over its leading dimension")
            period = xc.numel() // D
        ctx.x_bcast = period > 0
        w = weight.detach().float().contiguous()
        b = bias.detach().float().contiguous() if bias is not None else None
        x_new = torch.empty(dc.shape, device=x.device, dtype=torch.float32)
        y = torch.empty(dc.shape, device=x.device, dtype=out_dtype)
        mean = None if rms else torch.empty(M, device=x.device, dtype=torch.float32)
        rstd = torch.empty(M, device=x.device, dtype=torch.float32)
        check(lib().fk_add_norm_forward(ptr(xc), ptr(dc), ptr(w), ptr(b), ptr(x_new), ptr(y), _DT[out_dtype], ptr(mean),
                                        ptr(rstd), M, D, float(eps), int(rms), period, stream()), "fk_add_norm_forward")
        ctx.save_for_backward(x_new, w, mean if mean is not None else torch.empty(0, device=x.device), rstd)
        ctx.rms, ctx.has_bias, ctx.w_dtype = rms, bias is not None, weight.dtype
        return x_new, y

    @staticmethod
    @on_tensor_device
    def backward(ctx, g_xnew, g_y):
        x_new, w, mean, rstd = ctx.saved_tensors
        D = x_new.shape[-1]
        M = x_new.numel() // D
        if g_y is None:
            g_y = torch.zeros(x_new.shape, device=x_new.device, dtype=torch.bfloat16)
        g_y = g_y.contiguous()
        if g_y.dtype not in _DT:
            g_y = g_y.float()
        if g_xnew is not None:
            g_xnew = g_xnew.contiguous().float()
        dx = torch.empty_like(x_new)
        dx16 = torch.empty(x_new.shape, device=x_new.device, dtype=torch.bfloat16)
        nb = lib().fk_norm_backward_grid()
        dwp = torch.empty(nb, D, device=x_new.device, dtype=torch.float32)
        dbp = torch.empty(nb, D, device=x_new.device, dtype=torch.float32) if ctx.has_bias else None
        check(lib().fk_add_norm_backward(ptr(x_new), ptr(g_y), _DT[g_y.dtype], ptr(g_xnew), ptr(w),
                                         ptr(mean) if not ctx.rms else 0, ptr(rstd), ptr(dx), ptr(dx16), ptr(dwp), ptr(dbp),
                                         M, D, int(ctx.rms), stream()), "fk_add_norm_backward")
        dw, db = _reduce_partials(dwp, dbp, ctx.w_dtype)
        if ctx.x_bcast:
            dx = dx.sum(0, keepdim=True)
        return dx, dx16, dw, db, None, None, None


def add_layer_norm(x, delta, weight, bias, eps=1e-5, out_dtype=torch.bfloat16):
    """x_new = x + delta; y = LayerNorm(x_new)  ->  (x_new fp32, y)."""
    return _AddNormFn.apply(x, delta, weight, bias, eps, False, out_dtype)


def add_rms_norm(x, delta, weight, eps=1e-6, out_dtype=torch.bfloat16):
    return _AddNormFn.apply(x, delta, weight, None, eps, True, out_dtype)


def layer_norm(x, weight, bias, eps=1e-5, out_dtype=torch.bfloat16):
    return _NormFn.apply(x, weight, bias, eps, False, out_dtype)


def rms_norm(x, weight, eps=1e-6, out_dtype=torch.bfloat16):
    return _NormFn.apply(x, weight, None, eps, True, out_dtype)


# ------------------------------------------------------------------------------------------------
# SwiGLU gate on the fused [.., 2H] projection
# ------------------------------------------------------------------------------------------------
class _SwiGLUFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, h13):
        require_cuda(h13)
        require_device()
        if h13.dtype != torch.bfloat16:
            raise FkError("swiglu expects the bf16 fused projection")
        h13 = h13.contiguous()
        H = h13.shape[-1] // 2
        M = h13.numel() // (2 * H)
        y = torch.empty(*h13.shape[:-1], H, device=h13.device, dtype=torch.bfloat16)
        check(lib().fk_swiglu_forward(ptr(h13), ptr(y), M, H, stream()), "fk_swiglu_forward")
        ctx.save_for_backward(h13)
        return y

    @staticmethod
    @on_tensor_device
    def backward(ctx, gy):
        (h13,) = ctx.saved_tensors
        H = h13.shape[-1] // 2
        M = h13.numel() // (2 * H)
        gy = gy.contiguous().to(torch.bfloat16)
        d = torch.empty_like(h13)
        check(lib().fk_swiglu_backward(ptr(h13), ptr(gy), ptr(d), M, H, stream()), "fk_swiglu_backward")
        return d


def swiglu(h13):
    return _SwiGLUFn.apply(h13)


# ------------------------------------------------------------------------------------------------
# mask labels and RoPE description
# ------------------------------------------------------------------------------------------------
class LabelMask:
    """key j visible to query i  <=>  kid[b, j] <= qid[b, i] (and, with a band, qid[b, i] - kid[b, j] < band).  Holds the
    per-tile label ranges, computed once and shared by every layer of a forward pass.

    band: optional int >= 1, a sliding window over labels (a query sees the keys of its own label and of the band - 1 labels
    before it).  Only `attention_kv` takes a banded mask; None is no band."""

    def __init__(self, qid: torch.Tensor, kid: Optional[torch.Tensor] = None, band: Optional[int] = None):
        self.band = _check_band(band)
        require_cuda(qid)
        self.qid = qid.to(torch.int32).contiguous()
        self.kid = self.qid if kid is None else kid.to(torch.int32).contiguous()
        self._pairs = None
        self.qmin, self.qmax = self._ranges(self.qid)
        if self.kid is self.qid:
            self.kmin, self.kmax = self.qmin, self.qmax
        else:
            self.kmin, self.kmax = self._ranges(self.kid)

    @staticmethod
    @on_tensor_device
    def _ranges(ids):
        B, S = ids.shape
        nt = (S + 63) // 64
        lo = torch.empty(B, nt, device=ids.device, dtype=torch.int32)
        hi = torch.empty(B, nt, device=ids.device, dtype=torch.int32)
        check(lib().fk_attn_label_ranges(ptr(ids), B, S, ptr(lo), ptr(hi), stream()), "fk_attn_label_ranges")
        return lo, hi

    @staticmethod
    def from_ranges(qid, kid, qmin, qmax, kmin, kmax, band: Optional[int] = None) -> "LabelMask":
        """labels whose per-tile ranges are already known (fk_stream_positions writes them with the labels)."""
        m = LabelMask.__new__(LabelMask)
        m.qid, m.kid, m.qmin, m.qmax, m.kmin, m.kmax, m._pairs = qid, kid, qmin, qmax, kmin, kmax, None
        m.band = _check_band(band)
        return m

    @staticmethod
    def block_causal(B: int, S: int, tokens_per_block: int, device) -> "LabelMask":
        """brainformer.py:93-111 build_advanced_causal_mask: attend iff block(k) <= block(q)."""
        ids = (torch.arange(S, device=device, dtype=torch.int32) // tokens_per_block)[None].expand(B, S)
        return LabelMask(ids.contiguous())

    @staticmethod
    def padding(is_padded: torch.Tensor) -> "LabelMask":
        """simple_mae:349-352: attend iff neither the query nor the key is a padded token."""
        big = torch.iinfo(torch.int32).max
        kid = torch.where(is_padded, big, 0).to(torch.int32)
        qid = torch.where(is_padded, -1, 0).to(torch.int32)
        return LabelMask(qid, kid)

    def visible_pairs(self) -> torch.Tensor:
        """number of (query, key) pairs the mask lets through, summed over the batch: a 0-dim device tensor (no host
        sync) -- the algorithmic work of the attention kernels for the per-launch roofline figures of bench.py."""
        if self._pairs is None:
            k_sorted = torch.sort(self.kid, dim=1)[0]
            self._pairs = torch.searchsorted(k_sorted, self.qid.contiguous(), right=True).sum(dtype=torch.float64)
        return self._pairs

    def dense(self) -> torch.Tensor:
        """[B, 1, Sq, Sk] bool, True = attend (only for tests / the library-SDPA compatibility path)."""
        vis = self.kid[:, None, None, :] <= self.qid[:, None, :, None]
        if self.band is not None:
            vis &= (self.qid.long()[:, None, :, None] - self.kid.long()[:, None, None, :]) < self.band
        return vis


def _check_band(band) -> Optional[int]:
    if band is None:
        return None
    try:
        band = operator.index(band)
    except TypeError:
        raise FkError(f"LabelMask: band must be an int >= 1 or None, got {band!r}") from None
    if band < 1:
        raise FkError(f"LabelMask: band must be >= 1, got {band}")
    return band


def _no_band(mask, what: str) -> None:
    if mask is not None and mask.band is not None:
        raise FkError(f"{what}: a banded LabelMask is taken by attention_kv only (no training or backward path has a band)")


# query label of a streamed slot past its row's count (fk_stream_positions_counts): no key label (>= 0) satisfies it
NO_LABEL = -2 ** 31


def stream_rows(rows, batch_size: int, what: str) -> list:
    """Row indices of a per-row stream reset as a list of ints: FkError for an index outside [0, batch_size) or a duplicate."""
    try:
        idx = [operator.index(r) for r in rows]
    except TypeError:
        raise FkError(f"{what}: rows must be a sequence of integer row indices, got {rows!r}") from None
    bad = [r for r in idx if not 0 <= r < batch_size]
    if bad:
        raise FkError(f"{what}: rows {bad} are outside the batch of {batch_size}")
    if len(set(idx)) != len(idx):
        raise FkError(f"{what}: rows {idx} name a row twice")
    return idx


def stream_length(lengths, what: str) -> int:
    """The one length of a stream whose rows are all at the same position; FkError once they differ."""
    if any(n != lengths[0] for n in lengths):
        raise FkError(f"{what}: the rows are at different positions ({list(lengths)}); read `lengths` instead")
    return lengths[0]


@on_tensor_device
def stream_positions(len_in: torch.Tensor, len_out: torch.Tensor, n_new: int, tokens_per_label: int, cap: int,
                     counts: Optional[torch.Tensor] = None):
    """One launch for the per-row bookkeeping of a streaming step whose rows sit at different positions: row b holds
    len_in[b] tokens (device int32 [B]) and appends n_new at positions p = len_in[b] + i.  Returns (qid [B, n_new] =
    p // tokens_per_label, qmin, qmax [B, ceil(n_new / 64)] its tile ranges, pos [B, n_new] = p, rows int64 [B * n_new] =
    b * cap + p) and writes len_out = len_in + n_new.

    counts: optional device int32 [B], the new tokens of each row (0 ... n_new): slots at or past counts[b] get the label
    INT_MIN, which sees no key, a RoPE position inside the table and the scratch row B * cap of a cache with B * cap + 1
    rows; len_out = len_in + counts."""
    require_cuda(len_in, len_out, counts)
    B = len_in.shape[0]
    if counts is not None and (counts.dtype != torch.int32 or counts.shape != (B,) or not counts.is_contiguous()):
        raise FkError(f"stream_positions: counts must be a contiguous int32 [{B}] tensor, got {counts.dtype} "
                      f"{tuple(counts.shape)}")
    dev = len_in.device
    qid = torch.empty(B, n_new, device=dev, dtype=torch.int32)
    nt = (n_new + 63) // 64
    qmin = torch.empty(B, nt, device=dev, dtype=torch.int32)
    qmax = torch.empty(B, nt, device=dev, dtype=torch.int32)
    pos = torch.empty(B, n_new, device=dev, dtype=torch.int32)
    rows = torch.empty(B * n_new, device=dev, dtype=torch.int64)
    check(lib().fk_stream_positions_counts(ptr(len_in), ptr(counts), ptr(len_out), B, n_new, tokens_per_label, cap, ptr(qid),
                                           ptr(qmin), ptr(qmax), ptr(pos), ptr(rows), stream()), "fk_stream_positions")
    return qid, qmin, qmax, pos, rows


@on_tensor_device
def stream_ring_positions(len_in: torch.Tensor, len_out: torch.Tensor, n_new: int, tokens_per_label: int, cap: int,
                          keys: LabelMask, inv_freq: torch.Tensor, counts: Optional[torch.Tensor] = None):
    """One launch for the per-row bookkeeping of a sliding streaming step over ring caches of `cap` tokens per row: row b
    holds len_in[b] tokens (device int64 [B], unbounded) and appends its new slots i < counts[b] (all n_new without counts)
    at positions p = len_in[b] + i.  Returns (qid [B, n_new] = p // tokens_per_label (NO_LABEL past a count), qmin, qmax its
    tile ranges, rows int64 [B * n_new] = b * cap + p mod cap (B * cap past a count), rope fp32 [B * n_new, hd/2, 2] the
    (cos, sin) of p * inv_freq computed in fp64), writes the key label p // tokens_per_label into ring slot p mod cap of
    keys.kid [B, cap] with the tile ranges keys.kmin / kmax of the tiles it wrote, and len_out = len_in + counts."""
    require_cuda(len_in, len_out, counts, inv_freq)
    B = len_in.shape[0]
    for t, shape, dt in ((len_in, (B,), torch.int64), (len_out, (B,), torch.int64), (counts, (B,), torch.int32),
                         (keys.kid, (B, cap), torch.int32)):
        if t is not None and (t.dtype != dt or t.shape != shape or not t.is_contiguous()):
            raise FkError(f"stream_ring_positions: expected a contiguous {dt} {shape} tensor, got {t.dtype} {tuple(t.shape)}")
    if inv_freq.dtype != torch.float32 or inv_freq.dim() != 1 or not inv_freq.is_contiguous():
        raise FkError("stream_ring_positions: inv_freq must be a contiguous fp32 vector")
    half = inv_freq.shape[0]
    dev = len_in.device
    qid = torch.empty(B, n_new, device=dev, dtype=torch.int32)
    nt = (n_new + 63) // 64
    qmin = torch.empty(B, nt, device=dev, dtype=torch.int32)
    qmax = torch.empty(B, nt, device=dev, dtype=torch.int32)
    rows = torch.empty(B * n_new, device=dev, dtype=torch.int64)
    rope = torch.empty(B * n_new, half, 2, device=dev, dtype=torch.float32)
    check(lib().fk_stream_ring_positions(ptr(len_in), ptr(counts), ptr(len_out), B, n_new, tokens_per_label, cap, ptr(qid),
                                         ptr(qmin), ptr(qmax), ptr(rows), ptr(keys.kid), ptr(keys.kmin), ptr(keys.kmax),
                                         ptr(inv_freq), half, ptr(rope), stream()), "fk_stream_ring_positions")
    return qid, qmin, qmax, rows, rope


def stream_counts(counts, batch_size: int, limit: int, unit: int, what: str) -> list:
    """Per-row counts of new data of a streaming step as a list of ints: FkError for a sequence that is not one int per
    row, or a count outside [0, limit] or not a multiple of `unit`; the message names the rows."""
    try:
        c = [operator.index(v) for v in counts]
    except TypeError:
        raise FkError(f"{what}: counts must be a sequence of {batch_size} ints, got {counts!r}") from None
    if len(c) != batch_size:
        raise FkError(f"{what}: {len(c)} counts for a batch of {batch_size} rows")
    bad = [b for b, v in enumerate(c) if not 0 <= v <= limit]
    if bad:
        raise FkError(f"{what}: counts {[c[b] for b in bad]} of rows {bad} are outside [0, {limit}]")
    bad = [b for b, v in enumerate(c) if v % unit]
    if bad:
        raise FkError(f"{what}: counts {[c[b] for b in bad]} of rows {bad} are not multiples of {unit}")
    return c


class RopeSpec:
    """table: fp32 [P, hd/2, 2] (cos, sin) = view_as_real(build_complex_rope_cache(...)); position of token
    (b, s) = pos[b, s] if pos is given else s + offset."""

    def __init__(self, table: torch.Tensor, pos: Optional[torch.Tensor] = None, offset: int = 0):
        self.table = table.contiguous()
        self.pos = None if pos is None else pos.to(torch.int32).contiguous()
        self.offset = int(offset)

    @staticmethod
    def from_complex(cache: torch.Tensor, T: int, last: bool = True) -> "RopeSpec":
        """cache [P, hd/2] complex64; brainformer slices rope[-T:] (last=True), simple_mae rope[:T]."""
        table = torch.view_as_real(cache).float().contiguous()
        return RopeSpec(table, None, cache.shape[0] - T if last else 0)


@on_tensor_device
def _rope_inplace(x4, spec: RopeSpec, inverse: bool):
    """x4: bf16 view [B, S, H, hd], hd 16, 32 or 64 (token stride arbitrary, head stride hd)."""
    B, S, H, hd = x4.shape
    assert x4.stride(3) == 1 and x4.stride(2) == hd
    check(lib().fk_rope(ptr(x4), x4.stride(0), x4.stride(1), B, S, H, hd, ptr(spec.table), spec.table.shape[0],
                        ptr(spec.pos), spec.offset, int(inverse), stream()), "fk_rope")


# ------------------------------------------------------------------------------------------------
# attention on the fused QKV projection
# ------------------------------------------------------------------------------------------------
_BWD_PARTS = (2, 4)     # diagnosis hook (scripts/gpu_attn_stalls.py profiles one backward kernel at a time)
_BWD_PROFILE = None     # diagnosis hook: (int64 counter tensor, mode) -> fk_attn_backward_tc_profile


class _AttnQKVFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, qkv, n_heads, rope, mask, scale, rope_applied=False):
        """qkv: bf16 [B, S, 3*H*hd] (hd 16, 32 or 64) fresh output of the fused projection (q|k|v); RoPE is applied in place unless the
        projection's epilogue already did it (rope_applied: the backward still rotates dq / dk back)."""
        require_cuda(qkv)
        require_device()
        _no_band(mask, "attention_qkv")        # (so its backward never sees a band either)
        if qkv.dtype != torch.bfloat16 or not qkv.is_contiguous():
            raise FkError("attention expects a contiguous bf16 QKV buffer")
        B, S, W = qkv.shape
        H = n_heads
        hd = W // (3 * H)
        v5 = qkv.view(B, S, 3, H, hd)
        q, k, v = v5[:, :, 0], v5[:, :, 1], v5[:, :, 2]
        rotate_here = rope is not None and not rope_applied
        if rotate_here:
            _rope_inplace(q, rope, False)
            _rope_inplace(k, rope, False)
        out = torch.empty(B, S, H * hd, device=qkv.device, dtype=torch.bfloat16)
        need_grad = qkv.requires_grad
        lse = torch.empty(B, H, S, device=qkv.device, dtype=torch.float32)
        m = mask
        margs = (ptr(m.qid) if m else 0, ptr(m.kid) if m else 0, ptr(m.qmin) if m else 0, ptr(m.qmax) if m else 0,
                 ptr(m.kmin) if m else 0, ptr(m.kmax) if m else 0, float(scale))
        # algorithmic flops of one score-shaped matmul over the visible pairs (only evaluated while bench.py's timer is on)
        qk = 0.0
        if _lib.TIMER.enabled:
            qk = (m.visible_pairs() if m else float(B) * S * S) * (2.0 * H * hd)
        ctx.qk_flops = qk
        if ATTN_FWD_IMPL == "legacy":
            with timed("attn_fwd", 2 * qk):
                check(lib().fk_attn_forward(ptr(q), ptr(k), ptr(v), ptr(out), ptr(lse), B, H, S, S, hd,
                                            q.stride(0), q.stride(1), k.stride(0), k.stride(1), v.stride(0), v.stride(1),
                                            out.stride(0), out.stride(1), *margs, stream()), "fk_attn_forward")
        else:
            with timed("attn_fwd", 2 * qk):
                check(lib().fk_attn_forward_tc(ptr(q), ptr(k), ptr(v), ptr(out), ptr(lse), B, H, S, hd,
                                               q.stride(0), q.stride(1), k.stride(0), k.stride(1), v.stride(0), v.stride(1),
                                               out.stride(0), out.stride(1), *margs, counters(_lib.CTR_ATTN_FWD), stream()),
                      "fk_attn_forward_tc")
        if rotate_here:
            ctx.mark_dirty(qkv)          # q and k were rotated in place: autograd's version counter must see the write
        ctx.save_for_backward(qkv, out, lse)
        ctx.rope, ctx.mask, ctx.scale, ctx.H = rope, mask, scale, H
        return out, (qkv if rotate_here else None)

    @staticmethod
    @on_tensor_device
    def backward(ctx, d_o, _d_qkv_rotated=None):
        qkv, out, lse = ctx.saved_tensors
        B, S, W = qkv.shape
        H = ctx.H
        hd = W // (3 * H)
        d_o = d_o.contiguous().to(torch.bfloat16)
        v5 = qkv.view(B, S, 3, H, hd)
        q, k, v = v5[:, :, 0], v5[:, :, 1], v5[:, :, 2]
        dqkv = torch.empty_like(qkv)
        d5 = dqkv.view(B, S, 3, H, hd)
        dq, dk, dv = d5[:, :, 0], d5[:, :, 1], d5[:, :, 2]
        delta = torch.empty(B, H, S, device=qkv.device, dtype=torch.float32)
        m = ctx.mask
        common = (ptr(m.qid) if m else 0, ptr(m.kid) if m else 0, ptr(m.qmin) if m else 0, ptr(m.qmax) if m else 0,
                  ptr(m.kmin) if m else 0, ptr(m.kmax) if m else 0, float(ctx.scale))

        work = {"attn_delta": 0.0, "attn_bwd_dkv": 4 * ctx.qk_flops, "attn_bwd_dq": 1 * ctx.qk_flops}

        def legacy(name, part):
            with timed(name, work[name]):
                check(lib().fk_attn_backward(ptr(q), ptr(k), ptr(v), ptr(out), ptr(d_o), ptr(lse), ptr(delta), ptr(dq), ptr(dk),
                                             ptr(dv), B, H, S, S, hd, q.stride(0), q.stride(1), k.stride(0), k.stride(1),
                                             v.stride(0), v.stride(1), out.stride(0), out.stride(1), d_o.stride(0), d_o.stride(1),
                                             dq.stride(0), dq.stride(1), dk.stride(0), dk.stride(1), dv.stride(0), dv.stride(1),
                                             *common, part, stream()), "fk_attn_backward")

        fold = ATTN_BWD_IMPL != "legacy" and ATTN_BWD_OPERANDS != "transposed" and ATTN_BWD_STATS == "folded"
        aug = None
        if fold:
            # delta and the statistics rows the score MMAs take as one more K step (lse / delta folded into the tensor core)
            aug = torch.empty(B, H, S, 16, device=qkv.device, dtype=torch.bfloat16)
            d4a = d_o.view(B, S, H, hd)
            with timed("attn_delta", 0.0):
                check(lib().fk_attn_aug(ptr(out), ptr(d4a), ptr(lse), ptr(delta), ptr(aug), B, H, S, hd, out.stride(0), out.stride(1),
                                        d4a.stride(0), d4a.stride(1), float(ctx.scale), stream()), "fk_attn_aug")
        else:
            legacy("attn_delta", 1)
        rope_done = False
        r = ctx.rope
        rope_args = (ptr(r.table), r.table.shape[0], ptr(r.pos), r.offset) if r is not None else (0, 0, 0, 0)
        if ATTN_BWD_IMPL == "legacy":
            legacy("attn_bwd_dkv", 2)
            legacy("attn_bwd_dq", 4)
        else:
            # tcgen05 path
            Sp = (S + 7) // 8 * 8
            d4 = d_o.view(B, S, H, hd)
            tr = {"q": None, "k": None, "do": None}
            if ATTN_BWD_OPERANDS == "transposed":
                # K-major (token-contiguous) copies of q, k, dO for the contractions over tokens; the default reads the
                # [tokens][32] tiles MN-major instead and needs no copies
                with timed("attn_transpose"):
                    for name, src in (("q", q), ("k", k), ("do", d4)):
                        t = torch.empty(B, H, hd, Sp, device=qkv.device, dtype=torch.bfloat16)
                        check(lib().fk_attn_transpose(ptr(src), src.stride(0), src.stride(1), B, S, H, hd, ptr(t), Sp, stream()),
                              "fk_attn_transpose")
                        tr[name] = t
            for name, part in (("attn_bwd_dkv", 2), ("attn_bwd_dq", 4)):
                if part not in _BWD_PARTS:
                    continue
                args = (ptr(q), ptr(k), ptr(v), ptr(d4), ptr(tr["q"]), ptr(tr["k"]), ptr(tr["do"]), Sp,
                        ptr(lse), ptr(delta), ptr(aug), ptr(dq), ptr(dk), ptr(dv), B, H, S, hd,
                        q.stride(0), q.stride(1), k.stride(0), k.stride(1), v.stride(0), v.stride(1),
                        d4.stride(0), d4.stride(1), dq.stride(0), dq.stride(1), dk.stride(0),
                        dk.stride(1), dv.stride(0), dv.stride(1), *common, *rope_args, part, counters(_lib.CTR_ATTN_BWD))
                with timed(name, work[name]):
                    if _BWD_PROFILE is not None:
                        check(lib().fk_attn_backward_tc_profile(*args, ptr(_BWD_PROFILE[0]), int(_BWD_PROFILE[1]), stream()),
                              "fk_attn_backward_tc_profile")
                    else:
                        check(lib().fk_attn_backward_tc(*args, stream()), "fk_attn_backward_tc")
            rope_done = True                          # dq / dk were rotated back inside the kernels
        if ctx.rope is not None and not rope_done:
            _rope_inplace(dq, ctx.rope, True)
            _rope_inplace(dk, ctx.rope, True)
        return dqkv, None, None, None, None, None


def _check_head_dim(hd: int) -> None:
    if hd not in (16, 32, 64):
        raise FkError("the attention kernels are built for head_dim 16, 32 and 64")
    if hd != 32:
        # the cross-check paths (mma.sync kernels, transposed operands, staged statistics) exist at head_dim 32 only
        for name, value, default in (("ATTN_FWD_IMPL", ATTN_FWD_IMPL, "tc"), ("ATTN_BWD_IMPL", ATTN_BWD_IMPL, "tc"),
                                     ("ATTN_BWD_OPERANDS", ATTN_BWD_OPERANDS, "mn"), ("ATTN_BWD_STATS", ATTN_BWD_STATS, "folded")):
            if value != default:
                raise FkError(f"{name} = {value!r} is a head_dim-32 cross-check; head_dim {hd} runs the default path only")


def attention_qkv(qkv, n_heads: int, rope: Optional[RopeSpec] = None, mask: Optional[LabelMask] = None,
                  scale: Optional[float] = None, rope_applied: bool = False):
    """softmax(q k^T * scale + mask) v over the fused QKV buffer -> [B, S, H*hd] bf16, head_dim hd 16, 32 or 64."""
    hd = qkv.shape[-1] // (3 * n_heads)
    _check_head_dim(hd)
    if scale is None:
        scale = hd ** -0.5
    return _AttnQKVFn.apply(qkv, n_heads, rope, mask, scale, rope_applied)[0]


def _head_view(t: torch.Tensor, H: int, hd: int, what: str) -> torch.Tensor:
    """[B, S, H*hd] bf16 view -> [B, S, H, hd] view of the same memory (never a copy)."""
    if t.dim() != 3 or t.shape[-1] != H * hd or t.dtype != torch.bfloat16 or t.stride(2) != 1:
        raise FkError(f"attention_kv: {what} must be a bf16 [B, S, {H * hd}] view with contiguous columns, "
                      f"got {tuple(t.shape)} {t.dtype} strides {t.stride()}")
    if t.stride(0) % 8 != 0 or t.stride(1) % 8 != 0 or t.data_ptr() % 16 != 0:
        raise FkError(f"attention_kv: {what} strides {t.stride()} must keep 16-byte alignment")
    return t.as_strided((t.shape[0], t.shape[1], H, hd), (t.stride(0), t.stride(1), hd, 1))


@on_tensor_device
def attention_kv(q, k, v, n_heads: int, mask: Optional[LabelMask] = None, scale: Optional[float] = None):
    """Inference-only softmax(q k^T * scale + mask) v with queries and keys of different lengths (a streaming step's new
    tokens against a key / value cache): q [B, Sq, H*hd], k / v [B, Sk, H*hd] bf16 views with any 16-byte aligned batch and
    token strides (read in place, never copied) -> [B, Sq, H*hd] bf16.  head_dim 16, 32 or 64.  mask: LabelMask(qid [B, Sq],
    kid [B, Sk]), key j visible to query i iff kid[b, j] <= qid[b, i] (and qid[b, i] - kid[b, j] < mask.band with a band);
    a query that sees no key gives a zero row.  The key axis is split into chunks whose partial results are merged in chunk
    order (bit-reproducible); a banded mask always takes that split path (fk_attn_forward_kv_band_tc)."""
    require_cuda(q, k, v)
    require_device()
    if torch.is_grad_enabled() and (q.requires_grad or k.requires_grad or v.requires_grad):
        raise FkError("attention_kv is inference only (no backward): run it under torch.no_grad() or on detached tensors")
    B, Sq, W = q.shape
    Sk = k.shape[1]
    H = n_heads
    hd = W // H
    _check_head_dim(hd)
    if W != H * hd or k.shape != (B, Sk, W) or v.shape != (B, Sk, W):
        raise FkError(f"attention_kv: q {tuple(q.shape)}, k {tuple(k.shape)}, v {tuple(v.shape)} do not match {H} heads")
    if Sq < 1 or Sk < 1:
        raise FkError("attention_kv: empty query or key axis")
    if mask is not None and (mask.qid.shape != (B, Sq) or mask.kid.shape != (B, Sk)):
        raise FkError(f"attention_kv: mask labels {tuple(mask.qid.shape)} / {tuple(mask.kid.shape)} do not match "
                      f"queries ({B}, {Sq}) and keys ({B}, {Sk})")
    q4, k4, v4 = _head_view(q, H, hd, "q"), _head_view(k, H, hd, "k"), _head_view(v, H, hd, "v")
    dev = q.device
    nch = lib().fk_attn_kv_chunks(B, H, Sq, Sk, 0)
    band = None if mask is None else mask.band
    out = torch.empty(B, Sq, W, device=dev, dtype=torch.bfloat16)
    part_o = part_ml = None
    if nch > 1 or band is not None:
        part_o = torch.empty(B, H, nch, Sq, hd, device=dev, dtype=torch.float32)
        part_ml = torch.empty(B, H, nch, Sq, 2, device=dev, dtype=torch.float32)
    m = mask
    margs = (ptr(m.qid) if m else 0, ptr(m.kid) if m else 0, ptr(m.qmin) if m else 0, ptr(m.qmax) if m else 0,
             ptr(m.kmin) if m else 0, ptr(m.kmax) if m else 0)
    scale = float(hd ** -0.5 if scale is None else scale)
    strides = (q4.stride(0), q4.stride(1), k4.stride(0), k4.stride(1), v4.stride(0), v4.stride(1), out.stride(0), out.stride(1))
    with timed("attn_fwd_kv", 4.0 * B * H * Sq * Sk * hd):
        if band is None:
            check(lib().fk_attn_forward_kv_tc(ptr(q4), ptr(k4), ptr(v4), ptr(out), None, B, H, Sq, Sk, hd, *strides, *margs,
                                              scale, ptr(part_o), ptr(part_ml), nch, counters(_lib.CTR_ATTN_FWD), stream()),
                  "fk_attn_forward_kv_tc")
        else:
            check(lib().fk_attn_forward_kv_band_tc(ptr(q4), ptr(k4), ptr(v4), ptr(out), None, B, H, Sq, Sk, hd, *strides,
                                                   *margs, scale, ptr(part_o), ptr(part_ml), nch, band,
                                                   counters(_lib.CTR_ATTN_FWD), stream()), "fk_attn_forward_kv_band_tc")
    return out


# ------------------------------------------------------------------------------------------------
# attention with few queries (perceiver resampler: <= 64 queries, head_dim 16 / 32 / 64, no mask)
# ------------------------------------------------------------------------------------------------
SMALL_ATTN_MAX_Q = 64


def small_attention_supported(Tq: int, head_dim: int) -> bool:
    return Tq <= SMALL_ATTN_MAX_Q and head_dim in (16, 32, 64)


def _rows_ok(t: torch.Tensor) -> torch.Tensor:
    """dense bf16 [B, T, W]."""
    if t.dtype != torch.bfloat16:
        t = t.to(torch.bfloat16)
    return t.contiguous()           # (gradient buffers share the operands' strides; the tensors here are small or already dense)


class _SmallAttnFn(torch.autograd.Function):
    @staticmethod
    @on_tensor_device
    def forward(ctx, q, k, v, n_heads, scale, rope_table, rope_q0, rope_k0):
        require_cuda(q, k, v)
        require_device()
        q, k, v = _rows_ok(q), _rows_ok(k), _rows_ok(v)
        B, Tq, W = q.shape
        S = k.shape[1]
        H = n_heads
        hd = W // H
        if k.shape != (B, S, W) or v.shape != (B, S, W):
            raise FkError(f"small_attention: q {tuple(q.shape)}, k {tuple(k.shape)}, v {tuple(v.shape)} do not match")
        if not small_attention_supported(Tq, hd):
            raise FkError("small_attention serves <= 64 queries at head_dim 16 / 32 / 64")
        dev = q.device
        nch = lib().fk_small_attn_chunks(S)
        out = torch.empty(B, Tq, W, device=dev, dtype=torch.bfloat16)
        lse = torch.empty(B, H, Tq, device=dev, dtype=torch.float32)
        part_o = torch.empty(B, H, nch, Tq, hd, device=dev, dtype=torch.float32)
        part_ml = torch.empty(B, H, nch, Tq, 2, device=dev, dtype=torch.float32)
        rl = 0 if rope_table is None else rope_table.shape[0]
        with timed("small_attn_fwd", 4.0 * B * H * Tq * S * hd):
            check(lib().fk_small_attn_forward(ptr(q), q.stride(0), q.stride(1), ptr(k), k.stride(0), k.stride(1), ptr(v),
                                              v.stride(0), v.stride(1), ptr(out), out.stride(0), out.stride(1), ptr(lse), B, H,
                                              Tq, S, hd, scale, ptr(rope_table), rl, rope_q0, rope_k0, ptr(part_o),
                                              ptr(part_ml), None, stream()), "fk_small_attn_forward")
        ctx.save_for_backward(q, k, v, out, lse)
        ctx.meta = (H, hd, scale, rope_table, rope_q0, rope_k0, nch)
        return out

    @staticmethod
    @on_tensor_device
    def backward(ctx, g):
        q, k, v, out, lse = ctx.saved_tensors
        H, hd, scale, rope_table, rope_q0, rope_k0, nch = ctx.meta
        B, Tq, W = q.shape
        S = k.shape[1]
        g = _rows_ok(g)
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        if dk.stride() != k.stride() or dv.stride() != v.stride() or dq.stride() != q.stride():
            raise FkError("small_attention backward: gradient buffers must share the operands' strides")
        part_dq = torch.empty(B, H, nch, Tq, hd, device=q.device, dtype=torch.float32)
        rl = 0 if rope_table is None else rope_table.shape[0]
        with timed("small_attn_bwd", 10.0 * B * H * Tq * S * hd):
            check(lib().fk_small_attn_backward(ptr(q), q.stride(0), q.stride(1), ptr(k), k.stride(0), k.stride(1), ptr(v),
                                               v.stride(0), v.stride(1), ptr(out), out.stride(0), out.stride(1), ptr(g),
                                               g.stride(0), g.stride(1), ptr(lse), ptr(dq), ptr(dk), ptr(dv), B, H, Tq, S, hd,
                                               scale, ptr(rope_table), rl, rope_q0, rope_k0, ptr(part_dq), stream()),
                  "fk_small_attn_backward")
        return dq, dk, dv, None, None, None, None, None


class _SmallAttnKVFn(torch.autograd.Function):
    """small_attention on a FUSED key | value projection kv [B, S, 2 * H * hd] (columns [0, W) = k, [W, 2 W) = v): the kernels
    read the two halves in place through their row strides, and the backward writes dk | dv into ONE buffer of the same
    layout, so the projection that produced kv gets a single gradient (one dX GEMM, one dW GEMM, no gradient add)."""

    @staticmethod
    @on_tensor_device
    def forward(ctx, q, kv, n_heads, scale, rope_table, rope_q0, rope_k0):
        require_cuda(q, kv)
        require_device()
        q, kv = _rows_ok(q), _rows_ok(kv)
        B, Tq, W = q.shape
        S = kv.shape[1]
        H = n_heads
        hd = W // H
        if kv.shape != (B, S, 2 * W) or kv.stride(2) != 1:
            raise FkError(f"small_attention_kv: q {tuple(q.shape)} and kv {tuple(kv.shape)} do not match")
        if not small_attention_supported(Tq, hd):
            raise FkError("small_attention serves <= 64 queries at head_dim 16 / 32 / 64")
        k, v = kv[..., :W], kv[..., W:]
        dev = q.device
        nch = lib().fk_small_attn_chunks(S)
        out = torch.empty(B, Tq, W, device=dev, dtype=torch.bfloat16)
        lse = torch.empty(B, H, Tq, device=dev, dtype=torch.float32)
        part_o = torch.empty(B, H, nch, Tq, hd, device=dev, dtype=torch.float32)
        part_ml = torch.empty(B, H, nch, Tq, 2, device=dev, dtype=torch.float32)
        rl = 0 if rope_table is None else rope_table.shape[0]
        with timed("small_attn_fwd", 4.0 * B * H * Tq * S * hd):
            check(lib().fk_small_attn_forward(ptr(q), q.stride(0), q.stride(1), ptr(k), k.stride(0), k.stride(1), ptr(v),
                                              v.stride(0), v.stride(1), ptr(out), out.stride(0), out.stride(1), ptr(lse), B, H,
                                              Tq, S, hd, scale, ptr(rope_table), rl, rope_q0, rope_k0, ptr(part_o),
                                              ptr(part_ml), None, stream()), "fk_small_attn_forward")
        ctx.save_for_backward(q, kv, out, lse)
        ctx.meta = (H, hd, scale, rope_table, rope_q0, rope_k0, nch)
        return out

    @staticmethod
    @on_tensor_device
    def backward(ctx, g):
        q, kv, out, lse = ctx.saved_tensors
        H, hd, scale, rope_table, rope_q0, rope_k0, nch = ctx.meta
        B, Tq, W = q.shape
        S = kv.shape[1]
        g = _rows_ok(g)
        k, v = kv[..., :W], kv[..., W:]
        dq = torch.empty_like(q)
        dkv = torch.empty(B, S, 2 * W, device=kv.device, dtype=kv.dtype)
        dk, dv = dkv[..., :W], dkv[..., W:]
        # (q and kv were made dense by _rows_ok in forward, so the fresh gradient buffers share their strides)
        part_dq = torch.empty(B, H, nch, Tq, hd, device=q.device, dtype=torch.float32)
        rl = 0 if rope_table is None else rope_table.shape[0]
        with timed("small_attn_bwd", 10.0 * B * H * Tq * S * hd):
            check(lib().fk_small_attn_backward(ptr(q), q.stride(0), q.stride(1), ptr(k), k.stride(0), k.stride(1), ptr(v),
                                               v.stride(0), v.stride(1), ptr(out), out.stride(0), out.stride(1), ptr(g),
                                               g.stride(0), g.stride(1), ptr(lse), ptr(dq), ptr(dk), ptr(dv), B, H, Tq, S, hd,
                                               scale, ptr(rope_table), rl, rope_q0, rope_k0, ptr(part_dq), stream()),
                  "fk_small_attn_backward")
        return dq, dkv, None, None, None, None, None


def small_attention_kv(q, kv, n_heads: int, scale: Optional[float] = None):
    """softmax(q k^T * scale) v with k | v given as one fused projection kv [B, S, 2 * H * hd] (no mask, no RoPE)."""
    hd = q.shape[-1] // n_heads
    if not (q.is_cuda and kv.is_cuda):
        raise FkError("frankenstein_b200 kernels run on a B200 only (no CPU fallback)")
    return _SmallAttnKVFn.apply(q, kv, n_heads, float(hd ** -0.5 if scale is None else scale), None, 0, 0)


@on_tensor_device
def small_attention_kv_cached(q, kv, n_heads: int, scale: Optional[float] = None, k_len: Optional[torch.Tensor] = None):
    """Inference-only small_attention_kv against a key | value cache: kv [B, S, 2 * H * hd] bf16 is a view with any 16-byte
    aligned batch / token strides (e.g. the first S tokens of a longer cache), read in place, never copied.
    k_len: optional device int32 [B], the number of keys of each trial (trials of a cache at different lengths): key j of
    trial b takes part iff j < min(S, k_len[b]); keys past it are never read, and a trial with no key gives a zero row."""
    require_cuda(q, kv, k_len)
    require_device()
    if k_len is not None and (k_len.dtype != torch.int32 or k_len.shape != (q.shape[0],) or not k_len.is_contiguous()):
        raise FkError(f"small_attention_kv_cached: k_len must be a contiguous int32 [{q.shape[0]}] tensor, got "
                      f"{k_len.dtype} {tuple(k_len.shape)}")
    if torch.is_grad_enabled() and (q.requires_grad or kv.requires_grad):
        raise FkError("small_attention_kv_cached is inference only: run it under torch.no_grad()")
    q = _rows_ok(q)
    B, Tq, W = q.shape
    S = kv.shape[1]
    H = n_heads
    hd = W // H
    if kv.shape != (B, S, 2 * W) or kv.dtype != torch.bfloat16 or kv.stride(2) != 1 or kv.stride(0) % 8 or kv.stride(1) % 8:
        raise FkError(f"small_attention_kv_cached: q {tuple(q.shape)} and kv {tuple(kv.shape)} (strides {kv.stride()}) "
                      "do not match or are not 16-byte aligned bf16 rows")
    if not small_attention_supported(Tq, hd):
        raise FkError("small_attention serves <= 64 queries at head_dim 16 / 32 / 64")
    k, v = kv[..., :W], kv[..., W:]
    dev = q.device
    nch = lib().fk_small_attn_chunks(S)
    out = torch.empty(B, Tq, W, device=dev, dtype=torch.bfloat16)
    lse = torch.empty(B, H, Tq, device=dev, dtype=torch.float32)
    part_o = torch.empty(B, H, nch, Tq, hd, device=dev, dtype=torch.float32)
    part_ml = torch.empty(B, H, nch, Tq, 2, device=dev, dtype=torch.float32)
    scale = float(hd ** -0.5 if scale is None else scale)
    with timed("small_attn_fwd", 4.0 * B * H * Tq * S * hd):
        check(lib().fk_small_attn_forward(ptr(q), q.stride(0), q.stride(1), ptr(k), k.stride(0), k.stride(1), ptr(v),
                                          v.stride(0), v.stride(1), ptr(out), out.stride(0), out.stride(1), ptr(lse), B, H,
                                          Tq, S, hd, scale, None, 0, 0, 0, ptr(part_o), ptr(part_ml), ptr(k_len), stream()),
              "fk_small_attn_forward")
    return out


def small_attention(q, k, v, n_heads: int, scale: Optional[float] = None, rope: Optional[RopeSpec] = None,
                    rope_q0: Optional[int] = None, rope_k0: Optional[int] = None):
    """softmax(q k^T * scale) v for few queries: q [B, Tq <= 64, H*hd], k / v [B, S, H*hd] -> [B, Tq, H*hd] bf16 (no mask).
    rope: table positions of query t / key j are rope_q0 + t / rope_k0 + j (defaults: the spec's offset for both)."""
    hd = q.shape[-1] // n_heads
    if scale is None:
        scale = hd ** -0.5
    table = None
    if rope is not None:
        if rope.pos is not None:
            raise FkError("small_attention takes contiguous rope positions only")
        table = rope.table
        rope_q0 = rope.offset if rope_q0 is None else rope_q0
        rope_k0 = rope.offset if rope_k0 is None else rope_k0
    if not (q.is_cuda and k.is_cuda and v.is_cuda):
        raise FkError("frankenstein_b200 kernels run on a B200 only (no CPU fallback)")
    return _SmallAttnFn.apply(q, k, v, n_heads, float(scale), table, int(rope_q0 or 0), int(rope_k0 or 0))
