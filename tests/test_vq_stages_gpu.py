"""Float64 parity of every stage of the vector-quantiser training chain (csrc/vq_ops.cu): operand preparation, the
finish kernel (candidate merge, exact re-score, gather, straight-through output, commitment loss), backward, EMA
statistics, EMA finalize with Laplace smoothing and dead-code reset, the k-means mean update and the perplexity.

Each stage is fed the kernels' own upstream outputs (the indices `finish` returned, the `xn` `prepare_input` wrote,
the statistics `ema_stats` summed), so a bf16 near-tie that flips an assignment cannot blur an arithmetic comparison.
The references are written here in float64; the oracle (oracle/vector_quantize_ref.py) cannot serve, it computes in
fp32.  `test_references_match_oracle` (no GPU) ties the references to the oracle's semantics.

Bounds are fp32 error bounds of the kernels' own evaluation order, scaled by the magnitude of the terms a result is
formed from (never by the result, which may cancel, and never by a tensor-wide maximum).  U = 2^-24 is the unit
roundoff of fp32; a sum evaluated along a tree whose longest path has n additions is off by at most n * U * sum |terms|.
Where a kernel rounds once (gathers, bf16 casts, the straight-through expression, an fp32 division) the comparison is
bit equality with the same fp32 expression evaluated by PyTorch.
"""
import math
import random
import zlib

import pytest
import torch
import torch.nn.functional as F

from tests.helpers import make_vq_problem

U = 2.0 ** -24          # unit roundoff of fp32
SAFETY = 2.0            # the bounds below are first order; the factor covers the second-order terms
BN = 128                # code tile of the search kernel: c2pad is padded to a multiple of it
ROWS_PER_BLOCK = 8      # kRowsPerBlock of csrc/vq_ops.cu: rows per CTA of the finish kernel (one loss partial each)


def _round_up(a, b):
    return (a + b - 1) // b * b


def _f32(v):
    """the fp32 value the kernel receives for a Python float argument"""
    return float(torch.tensor(v, dtype=torch.float32))


def _gen(*key):
    return torch.Generator().manual_seed(zlib.crc32(repr(key).encode()))


def _fvq():
    from frankenstein_b200 import vector_quantize as fvq
    return fvq


def _assert_within(got, ref, tol, what):
    """|got - ref| <= SAFETY * tol elementwise (NaN fails)"""
    got, ref = got.double(), ref.double().to(got.device)
    tol = SAFETY * torch.as_tensor(tol, dtype=torch.float64, device=got.device).expand_as(ref)
    err = (got - ref).abs()
    bad = ~(err <= tol)
    if bad.any():
        where = tuple(bad.nonzero()[0].tolist())
        ratio = (err / tol.clamp_min(1e-300)).nan_to_num(float("inf")).max().item()
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound (worst err/bound "
                             f"{ratio:.3g}); first at {where}: got {got[where].item()!r}, ref {ref[where].item()!r}, "
                             f"bound {tol[where].item()!r}")


def _assert_bits(got, ref, what):
    if not torch.equal(got, ref):
        bad = (got != ref) & ~(torch.isnan(got) & torch.isnan(ref)) if got.is_floating_point() else got != ref
        where = tuple(bad.nonzero()[0].tolist()) if bad.any() else None
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements differ; first at {where}: "
                             f"got {got[where].item() if where else None!r}, ref {ref[where].item() if where else None!r}")


def _norm_rel(D):
    """relative error of an fp32 l2-normalisation as the kernels evaluate it, in units of U: the sum of squares runs
    ceil(D/32) serial steps per lane and 5 shuffle levels (+1 for the squares), the square root halves that and adds
    one rounding, the division adds one"""
    return ((D + 31) // 32 + 6) / 2.0 + 2.0


# ------------------------------------------------------------------------------------------------
# float64 references
# ------------------------------------------------------------------------------------------------
def ref_prepare_input(e, cosine):
    """(xn, inv_norm): F.normalize(e) and 1 / max(|e|, 1e-12) for cosine, (e, None) for Euclidean"""
    e = e.double()
    if not cosine:
        return e, None
    nrm = e.norm(dim=-1, keepdim=True).clamp_min(1e-12)
    return e / nrm, (1.0 / nrm).squeeze(-1)


def ref_c2(embed):
    """(|bf16(c)|^2, bound): the squares of bf16 values are exact in fp32; the sum runs Dp/32 serial steps per lane
    and 5 shuffle levels over positive terms"""
    D = embed.shape[1]
    b = embed.bfloat16().double()
    c2 = (b * b).sum(-1)
    return c2, (_round_up(D, 64) // 32 + 6) * U * c2


def ref_commitment_loss(xn, e_sel, w):
    """(w * mean((e[i] - x)^2), bound).  The kernel rounds e - x once and squares it (relative 3U per term), adds 4
    terms per float4 and ceil(D/128) float4 per lane, 8 levels of the block sum, one serial pass over
    ceil(blocks/256) partials and 8 more levels, then scales by an fp32 w/(N D) (2 roundings).  All terms are
    positive, so the bound is the path length times U times the result."""
    N, D = xn.shape
    d = e_sel.double() - xn.double()
    val = w * (d * d).mean()
    blocks = (N + ROWS_PER_BLOCK - 1) // ROWS_PER_BLOCK
    depth = 3 + 4 + (D + 127) // 128 + 8 + (blocks + 255) // 256 + 8 + 2
    return val, depth * U * abs(val)


def ref_backward(x, q, g_q, g_loss, w, cosine):
    """(dL/dx, bound) by float64 autograd of the oracle's expression: xn = normalize(x) (cosine) or x,
    out = xn + (q - xn).detach(), loss = w * mse(q, xn), L = <g_q, out> + g_loss * loss.

    Bound: v = g_q + g_loss * 2w/(N D) * (xn - q) is formed from terms of size vmag = |g_q| + |gl| (|xn| + |q|) with
    5 roundings (the coefficient twice, the difference, the product, the add).  Cosine adds the tangent projection
    (v - xn <xn, v>) / |x|: the dot product runs D/32 serial steps per lane + 5 shuffle levels over |v||xn|, and xn /
    inv_norm are themselves off by _norm_rel(D) U each; (D/32 + 32) U covers all of it."""
    N, D = x.shape
    x64 = x.double().requires_grad_(True)
    xn = F.normalize(x64, dim=-1) if cosine else x64
    q64 = q.double()
    out = xn + (q64 - xn).detach()
    loss = w * F.mse_loss(q64, xn)
    total = 0.0
    if g_q is not None:
        total = total + (out * g_q.double()).sum()
    if g_loss is not None:
        total = total + loss * g_loss
    total.backward()
    n = xn.detach()
    gl = abs(g_loss) * 2.0 * abs(w) / (N * D) if g_loss is not None else 0.0
    vmag = gl * (n.abs() + q64.abs())
    if g_q is not None:
        vmag = vmag + g_q.double().abs()
    if cosine:
        inv = 1.0 / x64.detach().norm(dim=-1, keepdim=True).clamp_min(1e-12)
        tol = (D / 32 + 32) * U * inv * (vmag + n.abs() * (vmag * n.abs()).sum(-1, keepdim=True))
    else:
        tol = 8 * U * vmag
    return x64.grad, tol


def _segsum_depth(ind, K, N):
    """longest addition path of vq_ema_segsum*: a code with c <= 32 rows is summed serially by one warp; up to 1024 rows
    32 warps sum ceil(c/32) rows each and the 32 partials are added serially; beyond, warp w sums the rows of this code
    that fall in its 32nd of the row range, then the 32 partials"""
    count = torch.bincount(ind, minlength=K)
    depth = count.double()
    mid = (count > 32) & (count <= 1024)
    depth[mid] = torch.ceil(count[mid].double() / 32) + 32
    per = ((N + 31) // 32 + 31) // 32 * 32
    for k in (count > 1024).nonzero().flatten().tolist():
        rows = (ind == k).nonzero().flatten()
        depth[k] = float(torch.bincount(rows // per).max()) + 32
    return depth


def ref_ema_stats(xn, ind, K):
    """(embed_sum, bound, bins): fp64 index_add and bincount; the bound is the segmented sum's path length times U
    times sum |x| of the code's rows"""
    N, D = xn.shape
    x = xn.double()
    s = torch.zeros(K, D, dtype=torch.float64, device=x.device).index_add_(0, ind, x)
    mag = torch.zeros(K, D, dtype=torch.float64, device=x.device).index_add_(0, ind, x.abs())
    return s, _segsum_depth(ind, K, N)[:, None] * U * mag, torch.bincount(ind, minlength=K)


def ref_ema_update(s, bins, cs, avg, decay, eps, thr, cand, cosine):
    """float64 restatement of the EMA finalize (oracle: VectorQuantizeRef.forward's EMA block + _expire_codes) on the
    exact fp32 inputs.  s [K, D] embed_sum, bins [K], cs [K] cluster_size, avg [K, D] embed_avg; cand [R, D] the
    candidate rows for dead-code reset (the i-th expired code in ascending order takes row i mod R), None for no reset.
    Returns {name: (value, bound)} and the expired mask.

    Bounds: a lerp a + w (b - a) rounds three times, relative to |a| + w (|a| + |b|); w = 1 - decay is exact in fp32
    for decay in [0.5, 1].  The total is a block sum over ceil(K/1024) serial codes per thread + 10 shuffle levels.
    The smoothing (cs + eps) / (total + K eps) * total rounds 5 times and inherits the relative errors of cs + eps and
    (at most twice) of the total; embed = embed_avg / smoothed adds one rounding; cosine then normalises (_norm_rel),
    which moves an element by at most twice the row's norm-wise error relative to the row's norm."""
    K, D = avg.shape
    w = 1.0 - _f32(decay)
    eps, thr = _f32(eps), _f32(thr)
    s, b, cs, avg = s.double(), bins.double(), cs.double(), avg.double()
    cs_new = cs + w * (b - cs)
    tol_cs = 3 * U * (cs.abs() + w * (b.abs() + cs.abs()))
    total = cs_new.sum()
    tol_total = ((K + 1023) // 1024 + 11) * U * cs_new.abs().sum() + tol_cs.sum()
    smoothed = (cs_new + eps) / (total + K * eps) * total
    rel_sm = 5 * U + tol_cs / (cs_new + eps) + 2 * tol_total / total
    avg_new = avg + w * (s - avg)
    tol_avg = 3 * U * (avg.abs() + w * (s.abs() + avg.abs()))
    e = avg_new / smoothed[:, None]
    tol_e = e.abs() * (rel_sm[:, None] + U) + tol_avg / smoothed[:, None]
    if cosine:
        nrm = e.norm(dim=-1, keepdim=True)
        n = e / nrm.clamp_min(1e-12)
        tol_e = n.abs() * _norm_rel(D) * U + 2 * tol_e.norm(dim=-1, keepdim=True) / nrm
        e = n
    expired = (cs_new < thr) if (cand is not None and thr > 0) else torch.zeros(K, dtype=torch.bool, device=cs.device)
    cs_out, tol_cs_out = cs_new.clone(), tol_cs.clone()
    if expired.any():
        rank = torch.cumsum(expired.long(), 0) - 1
        v = cand.double()[rank[expired] % cand.shape[0]]
        tol_v = torch.zeros_like(v)
        if cosine:
            v = v / v.norm(dim=-1, keepdim=True).clamp_min(1e-12)
            tol_v = v.abs() * _norm_rel(D) * U
        e[expired], tol_e[expired] = v, tol_v
        avg_new[expired], tol_avg[expired] = v * thr, thr * tol_v + U * (v * thr).abs()
        cs_out[expired], tol_cs_out[expired] = thr, 0.0
    return {"cluster_size": (cs_out, tol_cs_out), "embed_avg": (avg_new, tol_avg), "embed": (e, tol_e),
            "total": (total, tol_total), "cs_lerp": (cs_new, tol_cs)}, expired


def ref_kmeans_update(s, bins, means, cosine):
    """upstream `kmeans` mean update: sum / bins (one fp32 division), l2-normalised for cosine; a code without rows
    keeps its old mean"""
    D = means.shape[1]
    b = bins.double()
    new = s.double() / b.clamp_min(1)[:, None]
    tol = U * new.abs()
    if cosine:
        nrm = new.norm(dim=-1, keepdim=True)
        n = new / nrm.clamp_min(1e-12)
        tol = n.abs() * _norm_rel(D) * U + 2 * tol.norm(dim=-1, keepdim=True) / nrm.clamp_min(1e-300)
        new = n
    keep = (b == 0)[:, None]
    return torch.where(keep, means.double(), new), torch.where(keep, torch.zeros_like(tol), tol)


def ref_perplexity(ind, K):
    """(exp(-sum p log(p + 1e-10)), bound).  Per code the kernel rounds p = bins * fp32(1/N) twice, p + 1e-10 once,
    logf (1 ulp) and the product once: <= 6 U p (|log| + 1); the block sum adds ceil(K/1024) + 10 levels over
    sum |p log|; expf adds 2 ulp."""
    N = ind.numel()
    p = torch.bincount(ind, minlength=K).double() / N
    lg = torch.log(p + 1e-10)
    s = -(p * lg).sum()
    val = torch.exp(s)
    mag = (p * (lg.abs() + 1)).sum()
    return val, val * (((K + 1023) // 1024 + 10 + 6) * U * mag + 4 * U)


# ------------------------------------------------------------------------------------------------
# the references against the fp32 oracle (no GPU)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cosine", [False, True])
@pytest.mark.parametrize("N,K,D", [(96, 16, 12), (50, 40, 68)])
def test_references_match_oracle(N, K, D, cosine):
    """loss, input gradient (g_q and g_loss separately), EMA state with dead-code reset and the k-means update of the
    float64 references above agree with oracle/vector_quantize_ref.py to fp32 round-off"""
    from oracle import vector_quantize_ref as ovq
    w, g_loss, decay, eps, thr = 0.25, 3.0, 0.8, 1e-3, 2.0
    X, C = make_vq_problem(N, K, D, seed=N + K, cosine=cosine, noise=0.5)
    g = _gen("oracle", N, K, D, cosine)
    cs0 = torch.rand(K, generator=g) * 4
    cs0[:3] = torch.tensor([0.0, 1e-6, 3e-5])          # near zero: the Laplace smoothing's eps matters
    rows = torch.randperm(N, generator=g)
    gq = torch.randn(N, D, generator=g)
    ref = ovq.VectorQuantizeRef(dim=D, codebook_size=K, commitment_weight=w, use_cosine_sim=cosine, decay=decay, eps=eps,
                                threshold_ema_dead_code=thr,
                                sample_fn=lambda s, n, generator=None: rows[torch.arange(n) % N]).train()
    ref._codebook.embed.copy_(C[None]); ref._codebook.embed_avg.copy_((C * cs0[:, None])[None])
    ref._codebook.cluster_size.copy_(cs0[None])
    avg0 = ref._codebook.embed_avg[0].clone()
    x = X.clone().requires_grad_(True)
    q, ind, loss = ref(x)
    gx_q, = torch.autograd.grad((q * gq).sum(), x, retain_graph=True)
    gx_l, = torch.autograd.grad(g_loss * loss.sum(), x)
    # fp32 round-off of the oracle's own arithmetic, on top of the references' bounds for the kernels
    rt = 1e-5
    xn32 = F.normalize(X, dim=-1) if cosine else X
    lval, ltol = ref_commitment_loss(xn32, C[ind], w)
    _assert_within(loss.reshape(()), lval, ltol + rt * lval, "loss")
    for gq_, gl_, got, what in ((gq, None, gx_q, "grad (g_q)"), (None, g_loss, gx_l, "grad (g_loss)")):
        gval, gtol = ref_backward(X, C[ind], gq_, gl_, w, cosine)
        _assert_within(got, gval, 4 * gtol + rt * gval.abs(), what)
    s, _, bins = ref_ema_stats(xn32, ind, K)
    assert ref.last_expired is not None and ref.last_expired.any()
    out, expired = ref_ema_update(s, bins, cs0, avg0, decay, eps, thr, xn32[rows], cosine)
    assert torch.equal(expired, ref.last_expired)
    for name in ("cluster_size", "embed_avg", "embed"):
        val, tol = out[name]
        _assert_within(getattr(ref._codebook, name)[0], val, 4 * tol + rt * val.abs(), name)
    # k-means: one iteration from the first K rows
    init = torch.arange(K)
    means, kbins = ovq.kmeans(xn32, K, 1, cosine, init)
    dists = xn32 @ xn32[init].t() if cosine else -ovq.cdist(xn32[None], xn32[init][None])[0]
    buckets = dists.argmax(dim=-1)
    ks, _, kb = ref_ema_stats(xn32, buckets, K)
    assert torch.equal(kb, kbins)
    kval, ktol = ref_kmeans_update(ks, kb, xn32[init], cosine)
    _assert_within(means, kval, 4 * ktol + rt * kval.abs(), "kmeans means")


# ------------------------------------------------------------------------------------------------
# stages on the GPU
# ------------------------------------------------------------------------------------------------
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


@pytest.mark.gpu
@pytest.mark.parametrize("cosine", [False, True], ids=["euclid", "cosine"])
@pytest.mark.parametrize("D", [4, 68, 192, 256])
@pytest.mark.parametrize("dt", list(DTYPES))
def test_prepare_input(dt, D, cosine):
    """xn (Euclidean: the input itself, bit for bit; cosine: F.normalize within _norm_rel ulp), inv_norm, and the
    zero-padded bf16 operand == bf16(xn); a zero row and a row below the 1e-12 clamp; N = 1"""
    fvq = _fvq()
    g = _gen("prep", dt, D, cosine)
    for N in (1, 37):
        e = torch.randn(N, D, generator=g) * 10.0 ** (torch.rand(N, 1, generator=g) * 4 - 2)
        if N > 1:
            e[3] = 0.0                      # the eps clamp of F.normalize: xn = 0, inv_norm = 1e12
            e[5] *= 1e-14 / e[5].norm()     # |e| below the clamp (bf16 keeps it, f16 flushes it to 0)
        e = e.to(DTYPES[dt]).cuda()
        xn, xb, inv = fvq.prepare_input(e, cosine)
        Dp = _round_up(D, 64)
        assert xn.dtype == torch.float32 and xn.shape == (N, D) and xb.shape == (N, Dp)
        if cosine:
            rxn, rinv = ref_prepare_input(e, True)
            _assert_within(xn, rxn, _norm_rel(D) * U * rxn.abs(), "xn")
            _assert_within(inv, rinv, _norm_rel(D) * U * rinv.abs(), "inv_norm")
        else:
            assert inv is None
            _assert_bits(xn, e.float(), "xn")
        _assert_bits(xb[:, :D], xn.bfloat16(), "x_bf16")
        _assert_bits(xb[:, D:], torch.zeros_like(xb[:, D:]), "x_bf16 padding")


@pytest.mark.gpu
@pytest.mark.parametrize("cosine", [False, True], ids=["euclid", "cosine"])
@pytest.mark.parametrize("D", [4, 68, 192, 256])
@pytest.mark.parametrize("K", [1, 127, 128, 8192])
def test_prepare_codebook(K, D, cosine):
    fvq = _fvq()
    g = _gen("cb", K, D, cosine)
    embed = (torch.randn(K, D, generator=g) * 10.0 ** (torch.rand(K, 1, generator=g) * 4 - 2)).cuda()
    cb, c2pad = fvq.prepare_codebook(embed, cosine)
    Dp, Kpad = _round_up(D, 64), _round_up(K, BN)
    assert cb.shape == (K, Dp) and c2pad.shape == (Kpad,)
    _assert_bits(cb[:, :D], embed.bfloat16(), "cb")
    _assert_bits(cb[:, D:], torch.zeros_like(cb[:, D:]), "cb padding")
    if cosine:
        _assert_bits(c2pad[:K], torch.zeros(K, device="cuda"), "c2pad (cosine)")
    else:
        c2, tol = ref_c2(embed)
        _assert_within(c2pad[:K], c2, tol, "c2pad")
    assert torch.isposinf(c2pad[K:]).all()


# ---- finish on hand-built candidates --------------------------------------------------------------
def _finish_case(S, cosine, N=48, K=300, D=68):
    """Hand-built candidate slots [N, S, 4] and the index the finish kernel must pick.

    Each row holds valid (key, code) pairs -- keys equal to a base key, within 1e-6 of it, or 1..3 above it -- and
    junk the merge must skip: index -1, indices >= K or < -1, NaN and +inf keys, and copies of a valid pair (a pair
    is selected once).  Scenarios by row % 4: nothing valid (index 0); random; the two copies of a duplicated
    codeword with the higher index keyed first (equal exact scores: the lower index wins); more than 4 valid pairs with
    the row's nearest code keyed 5th (outside the 4 the merge keeps)."""
    rng = random.Random(zlib.crc32(repr(("finish", S, cosine)).encode()))
    g = _gen("finish", S, cosine)
    E = torch.randn(K, D, generator=g) / math.sqrt(D) * (0.5 + torch.rand(K, 1, generator=g))
    for i in range(8):
        E[K - 1 - 2 * i] = E[2 * i]
    X = torch.randn(N, D, generator=g) / math.sqrt(D)
    C = 4 * S
    cv = torch.empty(N, C)
    ci = torch.empty(N, C, dtype=torch.int32)
    expected = []
    ms = 32.0 / 512.0 / math.sqrt(D)
    for r in range(N):
        v0 = rng.uniform(-1.0, 1.0)
        scen = r % 4
        valid = []

        def rand_key():
            u = rng.random()
            return v0 if u < 0.3 else (v0 + rng.uniform(0, 1e-6) if u < 0.6 else v0 + rng.uniform(1.0, 3.0))

        if scen == 2 and C >= 4:
            i = rng.randrange(8)
            lo, hi = 2 * i, K - 1 - 2 * i
            X[r] = E[lo] + 0.01 * torch.randn(D, generator=g) / math.sqrt(D)
            valid += [(v0 - 2e-6, hi), (v0 - 1e-6, lo)]
            valid += [(rand_key(), rng.randrange(K)) for _ in range(rng.randint(0, C - 3))]
        elif scen == 3 and C >= 8:
            b = rng.randrange(K)
            X[r] = E[b] + 0.01 * torch.randn(D, generator=g) / math.sqrt(D)
            valid += [(v0, rng.randrange(K)) for _ in range(4)]
            valid += [(v0 + 1e-7, b)]
            valid += [(rand_key(), rng.randrange(K)) for _ in range(rng.randint(0, C - 6))]
        elif scen != 0:
            valid += [(rand_key(), rng.randrange(K)) for _ in range(rng.randint(1, C - 1))]
        valid = [(_f32(v), j) for v, j in valid]
        slots = list(valid)
        while len(slots) < C:
            kind = rng.randrange(7)
            if kind == 0:
                slots.append((rng.uniform(-100.0, -10.0), -1))
            elif kind == 1:
                slots.append((-100.0, K + rng.randrange(3)))
            elif kind == 2:
                slots.append((-100.0, rng.choice([-5, -(2 ** 31), 2 ** 31 - 1])))
            elif kind == 3:
                slots.append((float("nan"), rng.randrange(K)))
            elif kind == 4:
                slots.append((float("inf"), rng.randrange(K)))
            elif kind == 5 and valid:
                slots.append(rng.choice(valid))
            else:
                slots.append((-1000.0, -1))
        rng.shuffle(slots)
        cv[r] = torch.tensor([v for v, _ in slots])
        ci[r] = torch.tensor([j for _, j in slots], dtype=torch.int32)
        # expected: the 4 smallest distinct (key, index) pairs; re-score those within the margin of the best key
        sel = sorted(set(valid))[:4]
        if not sel:
            expected.append(0)
            continue
        x = X[r].double()
        xx = float(x @ x)

        def score(j):
            c = E[j].double()
            dot = float(x @ c)
            return -dot if cosine else math.sqrt(max(xx + float(c @ c) - 2 * dot, 0.0))

        c0 = E[sel[0][1]].double()
        margin = math.sqrt(xx * float(c0 @ c0)) * ms + abs(sel[0][0]) / 2048.0
        best, bs = sel[0][1], score(sel[0][1])
        scores = [(bs, best)]
        for v, j in sel[1:]:
            gap = v - sel[0][0]
            assert not (0.5 * margin < gap < 2 * margin), "setup: a key lies near the re-score margin"
            if gap > margin:
                break
            s = score(j)
            scores.append((s, j))
            if s < bs or (s == bs and j < best):
                best, bs = j, s
        for s, j in scores:     # setup: only copies of one codeword may tie in fp32
            assert j == best or torch.equal(E[j], E[best]) or abs(s - bs) > 1e-5 * (abs(bs) + 1e-3), "setup: near-tie"
        expected.append(best)
    return X, E, cv.view(N, S, 4), ci.view(N, S, 4), torch.tensor(expected, dtype=torch.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("cosine", [False, True], ids=["euclid", "cosine"])
@pytest.mark.parametrize("S", [1, 3, 40])
def test_finish_merges_hand_built_candidates(S, cosine):
    fvq = _fvq()
    X, E, cv, ci, expected = _finish_case(S, cosine)
    Xd, Ed = X.cuda(), E.cuda()
    ind, q, loss = fvq.finish(Xd, Ed, cv.cuda(), ci.cuda(), cosine, False, 0.25)
    _assert_bits(ind.cpu(), expected, "indices")
    _assert_bits(q, Ed[ind], "quantize (eval: the gathered codeword)")
    assert float(loss) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("D", [4, 68, 256])
@pytest.mark.parametrize("N", [1, 7, 9, 16384])
def test_finish_training(N, D):
    """straight-through output, commitment loss over a partial last block, the loss counter put back (a second call is
    bit-identical), and eval mode"""
    fvq = _fvq()
    K, w = 37, 0.25
    g = _gen("finish-train", N, D)
    xn = torch.randn(N, D, generator=g).cuda()
    E = (torch.randn(K, D, generator=g) * 1.5).cuda()
    idx = torch.randint(0, K, (N,), generator=g).cuda()
    cv = torch.zeros(N, 1, 4, device="cuda")
    ci = torch.full((N, 1, 4), -1, dtype=torch.int32, device="cuda")
    ci[:, 0, 0] = idx.int()
    ind, q, loss = fvq.finish(xn, E, cv, ci, False, True, w)
    _assert_bits(ind, idx, "indices")
    e = E[idx]
    _assert_bits(q, xn + (e - xn), "quantize (x + (e - x) in fp32)")
    lval, ltol = ref_commitment_loss(xn, e, w)
    _assert_within(loss.reshape(()), lval, ltol, "commitment loss")
    ind2, q2, loss2 = fvq.finish(xn, E, cv, ci, False, True, w)
    _assert_bits(loss2, loss, "loss of a repeated call")
    _assert_bits(q2, q, "quantize of a repeated call")
    ind3, q3, loss3 = fvq.finish(xn, E, cv, ci, False, False, w)
    _assert_bits(q3, e, "quantize (eval)")
    assert float(loss3) == 0.0


# ---- backward ------------------------------------------------------------------------------------
def _backward(fvq, g_q, g_loss, xn, q, inv, cosine, w):
    from frankenstein_b200._lib import check, lib, ptr, stream
    N, D = xn.shape
    ge = torch.empty(N, D, device="cuda")
    gl = None if g_loss is None else torch.tensor([g_loss], device="cuda")
    check(lib().fk_vq_backward(ptr(g_q), ptr(gl), ptr(xn), ptr(q), ptr(inv) if cosine else 0, N, D, int(cosine), w,
                               ptr(ge), stream()), "fk_vq_backward")
    return ge


@pytest.mark.gpu
@pytest.mark.parametrize("grads", ["g_q", "g_loss", "both"])
@pytest.mark.parametrize("D", [4, 68, 256])
@pytest.mark.parametrize("cosine", [False, True], ids=["euclid", "cosine"])
def test_backward(cosine, D, grads):
    """fk_vq_backward against float64 autograd; the g_loss-only case isolates the commitment term 2w/(N D) (x - q),
    which is 1e-5..1e-6 of an O(1) straight-through gradient when both are present"""
    fvq = _fvq()
    w = 0.25
    for N in (1, 13, 1003):
        g = _gen("bwd", cosine, D, grads, N)
        x = (torch.randn(N, D, generator=g) * 10.0 ** (torch.rand(N, 1, generator=g) * 2 - 1)).cuda()
        xn, _, inv = fvq.prepare_input(x, cosine)
        codes = torch.randn(N, D, generator=g).cuda()
        if cosine:
            codes = F.normalize(codes, dim=-1)
        q = xn + (codes - xn)                              # the straight-through value finish writes
        g_q = torch.randn(N, D, generator=g).cuda() if grads != "g_loss" else None
        g_loss = 3.0 if grads != "g_q" else None
        ge = _backward(fvq, g_q, g_loss, xn, q, inv, cosine, w)
        val, tol = ref_backward(x, q, g_q, g_loss, w, cosine)
        _assert_within(ge, val, tol, f"grad N={N}")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", ["f32", "bf16", "f16"])
@pytest.mark.parametrize("cosine", [False, True], ids=["euclid", "cosine"])
def test_module_backward_loss_only_and_half_inputs(cosine, dt):
    """through VectorQuantize: loss.backward() alone, and the gradient in the input's dtype (one rounding of the fp32
    gradient: one ulp of that dtype on top of the fp32 bound)"""
    fvq = _fvq()
    N, K, D, w = 203, 64, 68, 0.25
    X, C = make_vq_problem(N, K, D, seed=17, cosine=cosine, noise=0.5)
    m = fvq.VectorQuantize(dim=D, codebook_size=K, commitment_weight=w, use_cosine_sim=cosine).cuda().train()
    m._codebook.embed.copy_(C[None]); m._codebook.embed_avg.copy_(C[None]); m._codebook.cluster_size.fill_(1.0)
    m._mark_dirty(); m._kmeans_initted_host = True
    for loss_only in (True, False):
        x = X.to(DTYPES[dt]).cuda().requires_grad_(True)
        e_before = m._codebook.embed[0].clone()
        q, ind, loss = m(x[None])
        g_q = torch.randn(N, D, generator=_gen("mod-bwd", cosine, dt)).cuda()
        if loss_only:
            (2.0 * loss.sum()).backward()
        else:
            ((q[0] * g_q).sum() + 2.0 * loss.sum()).backward()
        assert x.grad.dtype == x.dtype
        val, tol = ref_backward(x.detach(), e_before[ind[0]], None if loss_only else g_q, 2.0, w, cosine)
        if dt == "f32":
            ulp = 0.0
        elif dt == "bf16":
            ulp = val.abs() * 2.0 ** -7 / SAFETY
        else:                                   # f16: relative below 2^-14 its subnormals are 2^-24 apart
            ulp = (val.abs() * 2.0 ** -10).clamp_min(2.0 ** -24) / SAFETY
        _assert_within(x.grad, val, tol + ulp, f"grad ({'loss only' if loss_only else 'both'})")


# ---- EMA statistics, finalize, k-means, perplexity ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("K,D", [(1025, 68), (8192, 256), (65536, 64)])
def test_ema_stats(K, D):
    """embed_sum and bins against fp64 index_add / bincount at K > 1024 (several codes per thread in the scan), with
    hot codes of 33, 1024, 1025 and 3000 rows (every segment path), the last code among them"""
    fvq = _fvq()
    N = 16384
    g = _gen("stats", K, D)
    xn = torch.randn(N, D, generator=g).cuda()
    ind = torch.randint(0, K, (N,), generator=g)
    hot = {K - 1: 33, 5: 1024, K // 2: 1025, 1000: 3000}
    ind[torch.isin(ind, torch.tensor(list(hot)))] = 7
    perm = torch.randperm(N, generator=g)
    at = 0
    for k, c in hot.items():
        ind[perm[at:at + c]] = k
        at += c
    ind = ind.cuda()
    stats = fvq.ema_stats(xn, ind, K)
    s, tol, bins = ref_ema_stats(xn, ind, K)
    for k, c in hot.items():
        assert int(bins[k]) == c
    _assert_bits(stats[K * D:], bins.float(), "bins")
    _assert_within(stats[:K * D].view(K, D), s, tol, "embed_sum")


def _ema_inputs(K, D, decay, thr, g):
    """cluster sizes with exact zeros and values near zero (where eps matters), integer bins, and no code whose
    updated cluster size lies within rounding of the threshold"""
    kind = torch.randint(0, 4, (K,), generator=g)
    cs = torch.rand(K, generator=g) * 6
    cs[kind == 0] = 0.0
    cs[kind == 1] = 10.0 ** (torch.rand(int((kind == 1).sum()), generator=g) * 4 - 8)
    bins = torch.randint(0, 8, (K,), generator=g).float() * (torch.rand(K, generator=g) < 0.6)
    if K == 1:
        cs[0], bins[0] = 0.5, 3.0
    if thr > 0:
        w = 1.0 - _f32(decay)
        near = ((cs.double() + w * (bins.double() - cs.double())) - thr).abs() < 1e-3
        cs[near] += 0.01
    avg = torch.randn(K, D, generator=g) * (cs[:, None] + 0.1)
    s = torch.randn(K, D, generator=g) * (bins[:, None] + 0.1)
    return cs, bins, avg, s


def _ema_update(fvq, stats, cs, avg, embed, D, cosine, decay, eps, thr, rows, xn):
    from frankenstein_b200._lib import check, lib, ptr, stream
    K = cs.numel()
    Dp, Kpad = _round_up(D, 64), _round_up(K, BN)
    cb = torch.empty(K, Dp, device="cuda", dtype=torch.bfloat16)
    c2pad = torch.empty(Kpad, device="cuda")
    total = torch.empty(1, device="cuda")
    rank = torch.empty(K, device="cuda", dtype=torch.int32)
    n_exp = torch.empty(1, device="cuda", dtype=torch.int32)
    check(lib().fk_vq_ema_update(ptr(stats), ptr(cs), ptr(avg), ptr(embed), K, D, Dp, Kpad, int(cosine), decay, eps, thr,
                                 ptr(rows), rows.numel(), ptr(xn), xn.shape[0], ptr(cb), ptr(c2pad), ptr(total),
                                 ptr(rank), ptr(n_exp), stream()), "fk_vq_ema_update")
    return cb, c2pad, total, rank, n_exp


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.0, 2.0])
@pytest.mark.parametrize("decay,eps", [(0.8, 1e-5), (0.99, 1e-5), (0.8, 1e-3)])
@pytest.mark.parametrize("cosine", [False, True], ids=["euclid", "cosine"])
@pytest.mark.parametrize("K,D", [(1, 68), (1000, 68), (1024, 256), (1025, 68), (8192, 256), (65536, 68)])
def test_ema_update(K, D, cosine, decay, eps, thr):
    """cluster_size lerp, its total, Laplace smoothing, embed_avg lerp, embed (cosine: normalised), the expired codes and
    their ranks, the candidate row each one takes (fewer and more candidates than expired codes), and the refreshed
    search operand == prepare_codebook(new embed)"""
    fvq = _fvq()
    g = _gen("ema", K, D, cosine, decay, eps, thr)
    cs, bins, avg, s = _ema_inputs(K, D, decay, thr, g)
    stats = torch.cat([s.reshape(-1), bins]).cuda()
    embed0 = torch.randn(K, D, generator=g).cuda()
    _, expired = ref_ema_update(s, bins, cs, avg, decay, eps, thr, torch.zeros(1, D), cosine)
    n_exp = int(expired.sum())
    for R in sorted({max(1, n_exp // 3), n_exp + 5}):
        src = torch.randn(max(64, 2 * R), D, generator=g)
        rows = torch.randperm(src.shape[0], generator=g)[:R]
        cs_d, avg_d, emb_d = cs.cuda(), avg.cuda(), embed0.clone()
        cb, c2pad, total, rank, n_exp_d = _ema_update(fvq, stats, cs_d, avg_d, emb_d, D, cosine, decay, eps, thr,
                                                      rows.cuda(), src.cuda())
        out, exp_ref = ref_ema_update(s, bins, cs, avg, decay, eps, thr, src[rows], cosine)
        what = f"R={R}"
        assert int(n_exp_d) == int(exp_ref.sum()), (what, int(n_exp_d), int(exp_ref.sum()))
        want_rank = torch.where(exp_ref, torch.cumsum(exp_ref.int(), 0) - 1, torch.full_like(exp_ref, -1, dtype=torch.int64))
        _assert_bits(rank.cpu().long(), want_rank, f"{what} expire ranks")
        _assert_within(total.reshape(()), *out["total"], f"{what} total")
        _assert_within(cs_d, *out["cluster_size"], f"{what} cluster_size")
        _assert_within(avg_d, *out["embed_avg"], f"{what} embed_avg")
        _assert_within(emb_d, *out["embed"], f"{what} embed")
        cb_ref, c2_ref = fvq.prepare_codebook(emb_d, cosine)
        _assert_bits(cb, cb_ref, f"{what} cb")
        _assert_bits(c2pad, c2_ref, f"{what} c2pad")


@pytest.mark.gpu
@pytest.mark.parametrize("cosine", [False, True], ids=["euclid", "cosine"])
@pytest.mark.parametrize("D", [68, 256])
@pytest.mark.parametrize("K", [64, 1025])
def test_kmeans_update(K, D, cosine):
    """sum / bins (cosine: normalised), the old mean kept where bins == 0, the operand refreshed"""
    from frankenstein_b200._lib import check, lib, ptr, stream
    fvq = _fvq()
    g = _gen("kmeans", K, D, cosine)
    N = 8 * K
    xn = torch.randn(N, D, generator=g).cuda()
    ind = torch.randint(0, K, (N,), generator=g)
    ind[ind % 7 == 3] = 0                      # codes 3, 10, 17, ... keep no rows
    ind = ind.cuda()
    stats = fvq.ema_stats(xn, ind, K)           # the kernel's own statistics
    means = torch.randn(K, D, generator=g).cuda()
    old = means.clone()
    Dp, Kpad = _round_up(D, 64), _round_up(K, BN)
    cb = torch.empty(K, Dp, device="cuda", dtype=torch.bfloat16)
    c2pad = torch.empty(Kpad, device="cuda")
    check(lib().fk_vq_kmeans_update(ptr(stats), ptr(means), K, D, Dp, Kpad, int(cosine), ptr(cb), ptr(c2pad), stream()),
          "fk_vq_kmeans_update")
    s, bins = stats[:K * D].view(K, D), stats[K * D:]
    assert (bins == 0).sum() >= K // 8
    val, tol = ref_kmeans_update(s, bins, old, cosine)
    if not cosine:
        _assert_bits(means, torch.where((bins == 0)[:, None], old, s / bins.clamp_min(1)[:, None]), "means")
    _assert_within(means, val, tol, "means")
    cb_ref, c2_ref = fvq.prepare_codebook(means, cosine)
    _assert_bits(cb, cb_ref, "cb")
    _assert_bits(c2pad, c2_ref, "c2pad")


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["uniform", "one-code", "random"])
@pytest.mark.parametrize("K", [1, 512, 8192])
def test_perplexity(K, pattern):
    from frankenstein_b200.vq_brain import perplexity
    g = _gen("perp", K, pattern)
    N = 4 * K + 3 if pattern == "random" else 4 * K
    if pattern == "uniform":
        ind = torch.arange(N) % K
    elif pattern == "one-code":
        ind = torch.full((N,), K - 1)
    else:
        ind = torch.randint(0, K, (N,), generator=g)
        ind[:K // 4 + 1] = K - 1
    val, tol = ref_perplexity(ind, K)
    got = perplexity(ind.cuda(), K)
    _assert_within(got.reshape(()), val, tol, "perplexity")
    if pattern == "uniform":
        assert abs(float(got) - K) <= 1e-4 * K


# ---- whole training steps ------------------------------------------------------------------------
MODULE_CASES = {"cfg4": dict(B=16, T=1024, K=8192, D=256, cosine=False),     # the default bench's quantiser
                "cfg1": dict(B=16, T=256, K=512, D=64, cosine=True)}        # the cosine VQ-VAE


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, "always"], ids=["in-stream", "side-stream"])
@pytest.mark.parametrize("cfg", list(MODULE_CASES))
def test_training_step_matches_float64(cfg, overlap):
    """two VectorQuantize training steps with dead-code reset: loss, straight-through output, input gradient, the EMA
    state, last_bins / last_n_expired and the search operand, each against the float64 reference from the module's
    state before the step, its indices and its xn"""
    fvq = _fvq()
    B, T, K, D, cosine = (MODULE_CASES[cfg][k] for k in ("B", "T", "K", "D", "cosine"))
    N, w, thr = B * T, 0.25, 2.0
    X, C = make_vq_problem(N, K, D, seed=K + D, cosine=cosine, noise=0.5)
    g = _gen("module", cfg)
    cs0 = 0.5 + torch.rand(K, generator=g) * 6
    m = fvq.VectorQuantize(dim=D, codebook_size=K, commitment_weight=w, use_cosine_sim=cosine,
                           threshold_ema_dead_code=thr).cuda().train()
    m._codebook.embed.copy_(C[None]); m._codebook.embed_avg.copy_((C * cs0[:, None])[None])
    m._codebook.cluster_size.copy_(cs0[None])
    m._mark_dirty(); m._kmeans_initted_host = True
    m.overlap_ema = overlap
    rows = torch.randperm(N, generator=g)
    m.sample_rows_override = rows
    R = min(K, N)
    for step in range(2):
        x = (X + 0.05 * torch.randn(X.shape, generator=g)).cuda()
        gq = torch.randn(N, D, generator=g).cuda()
        st = {k: v.clone() for k, v in m.state_dict().items()}
        xr = x.view(B, T, D).clone().requires_grad_(True)
        q, ind, loss = m(xr)
        ((q.view(N, D) * gq).sum() + 3.0 * loss.sum()).backward()
        sd = m.state_dict()                    # waits for an EMA update still running on the side stream
        cb, c2pad = m._operands()
        ind = ind.view(N)
        what = f"step {step}"
        e = st["_codebook.embed"][0][ind]
        xn = fvq.prepare_input(x, cosine)[0]
        _assert_bits(q.view(N, D), xn + (e - xn), f"{what} quantize")
        lval, ltol = ref_commitment_loss(xn, e, w)
        _assert_within(loss.reshape(()), lval, ltol, f"{what} loss")
        gval, gtol = ref_backward(x, e, gq, 3.0, w, cosine)
        _assert_within(xr.grad.view(N, D), gval, gtol, f"{what} input gradient")
        stats = fvq.ema_stats(xn, ind, K)
        s, bins = stats[:K * D].view(K, D), stats[K * D:]
        _assert_bits(m.last_bins, bins, f"{what} last_bins")
        _assert_bits(bins.long(), torch.bincount(ind, minlength=K), f"{what} bins")
        out, expired = ref_ema_update(s, bins, st["_codebook.cluster_size"][0], st["_codebook.embed_avg"][0], m.decay,
                                      m.eps, thr, xn[rows[:R].cuda()], cosine)
        cs_lerp, cs_tol = out["cs_lerp"]
        exact = bins.double() == st["_codebook.cluster_size"][0].double()       # the lerp is exact: cs + w * 0
        assert ((cs_lerp - thr).abs() > SAFETY * cs_tol).logical_or(exact).all(), \
            "setup: a cluster size lies within rounding of the threshold"
        assert 0 < int(expired.sum()) < K
        assert int(m.last_n_expired) == int(expired.sum()), (what, int(m.last_n_expired), int(expired.sum()))
        for name in ("cluster_size", "embed_avg", "embed"):
            _assert_within(sd["_codebook." + name][0], *out[name], f"{what} {name}")
        cb_ref, c2_ref = fvq.prepare_codebook(sd["_codebook.embed"][0].contiguous(), cosine)
        _assert_bits(cb, cb_ref, f"{what} cb")
        _assert_bits(c2pad, c2_ref, f"{what} c2pad")
