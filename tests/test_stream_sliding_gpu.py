"""Sliding streams (`Encoder.stream(..., sliding=True)`, `BrainFormer.stream(..., sliding=True)`): the banded split-key
attention (fk_attn_forward_kv_band_tc) against a float64 reference on ring-ordered labels, its exact invariants, the ring
bookkeeping kernel (fk_stream_ring_positions) against torch, and both streams over several windows against the fp32
oracle with a dense banded block-causal mask over the whole recording, with staggered sessions, filler, rejections and a
launch list that does not grow with the session's length.
"""
import random

import pytest
import torch

from tests.test_attention_masks_gpu import LSE_TOL, OUT_TOL
from tests.test_encoder_stream_gpu import CFG2, _counters_zero, _enc_cfg, _no_dense_attention, rel_close
from tests.test_stream_counts_gpu import _fill
from tests.test_stream_sessions_gpu import _brainformer

pytestmark = pytest.mark.gpu

LO, HI = -2 ** 31, 2 ** 31 - 1
NO_LABEL = LO
LN2 = 0.6931471805599453


# ------------------------------------------------------------------------------------------------
# banded attention kernel
# ------------------------------------------------------------------------------------------------
def _ring_labels(B, Sq, Sk, E, g, extreme=False):
    """ring-ordered labels: row b wrote positions P0 .. P0 + n - 1 of a recording into slots p mod Sk (label base + p // E),
    the other slots are INT_MAX; its queries are the last Sq positions (NO_LABEL before P0 and at ~10 % of the slots).
    extreme: row 0 labels end at INT_MAX - 1, row 1 start at INT_MIN + 1."""
    kid = torch.full((B, Sk), HI, dtype=torch.int64)
    qid = torch.full((B, Sq), NO_LABEL, dtype=torch.int64)
    for b in range(B):
        n = int(torch.randint(Sk // 2, Sk + 1, (1,), generator=g))
        P0 = int(torch.randint(0, 10 * Sk, (1,), generator=g))
        base = 0
        if extreme and b == 0:
            base = HI - 1 - (P0 + n) // E
        elif extreme and b == 1:
            base = LO + 1 - P0 // E
        p = torch.arange(P0, P0 + n)
        kid[b, p % Sk] = base + p // E
        qp = torch.arange(P0 + n - Sq, P0 + n)
        qid[b] = torch.where(qp >= P0, base + qp.div(E, rounding_mode="floor"), NO_LABEL)
    qid[torch.rand(B, Sq, generator=g) < 0.1] = NO_LABEL
    return qid.to(torch.int32).cuda(), kid.to(torch.int32).cuda()


def _visible(qid, kid, band):
    q, k = qid.long()[:, :, None], kid.long()[:, None, :]
    return (k <= q) & (q - k < band)                          # [B, Sq, Sk]


def _launch_band(q, k, v, H, labels, n_chunks, band, lse=True):
    """raw fk_attn_forward_kv_band_tc (band None: fk_attn_forward_kv_tc); returns (rc, out, lse)."""
    from frankenstein_b200 import _lib, ops
    from frankenstein_b200._lib import counters, lib, ptr, stream
    B, Sq, W = q.shape
    Sk = k.shape[1]
    hd = W // H
    m = ops.LabelMask(*labels)
    out = torch.zeros(B, Sq, W, device=q.device, dtype=torch.bfloat16)
    ls = torch.zeros(B, H, Sq, device=q.device, dtype=torch.float32) if lse else None
    part_o = torch.empty(B, H, n_chunks, Sq, hd, device=q.device, dtype=torch.float32)
    part_ml = torch.empty(B, H, n_chunks, Sq, 2, device=q.device, dtype=torch.float32)
    args = (ptr(q), ptr(k), ptr(v), ptr(out), ptr(ls), B, H, Sq, Sk, hd, q.stride(0), q.stride(1), k.stride(0), k.stride(1),
            v.stride(0), v.stride(1), out.stride(0), out.stride(1), ptr(m.qid), ptr(m.kid), ptr(m.qmin), ptr(m.qmax),
            ptr(m.kmin), ptr(m.kmax), float(hd ** -0.5), ptr(part_o), ptr(part_ml), n_chunks)
    if band is None:
        rc = lib().fk_attn_forward_kv_tc(*args, counters(_lib.CTR_ATTN_FWD), stream())
    else:
        rc = lib().fk_attn_forward_kv_band_tc(*args, band, counters(_lib.CTR_ATTN_FWD), stream())
    return rc, out, ls


def _operands(B, Sq, Sk, H, hd, g):
    q = (torch.randn(B, Sq, H * hd, generator=g) * 1.5).to(torch.bfloat16).cuda()
    k = (torch.randn(B, Sk, H * hd, generator=g) * 1.5).to(torch.bfloat16).cuda()
    v = torch.randn(B, Sk, H * hd, generator=g).to(torch.bfloat16).cuda()
    return q, k, v


def _check_band(out, lse, q, k, v, H, labels, band, what):
    B, Sq, W = q.shape
    hd = W // H
    vis = _visible(*labels, band)
    q4, k4, v4 = (t.view(B, -1, H, hd).double() for t in (q, k, v))
    s = torch.einsum("bqhd,bkhd->bhqk", q4, k4) * hd ** -0.5
    s = s.masked_fill(~vis[:, None], float("-inf"))
    ref = torch.einsum("bhqk,bkhd->bqhd", torch.softmax(s, -1).nan_to_num(0.0), v4)
    o = out.view(B, Sq, H, hd).double()
    vabs = v4.abs().amax(-1)                                   # [B, Sk, H]
    vmax = (vis[..., None].double() * vabs[:, None]).amax(2)   # [B, Sq, H]: the largest visible |v|
    err = (o - ref).abs().amax(-1)
    assert bool((err <= OUT_TOL * vmax + 1e-6).all()), f"{what}: out error {float((err / (vmax + 1e-30)).max()):.3g}"
    empty = ~vis.any(-1)
    assert bool((o[empty] == 0).all()), f"{what}: rows that see no key are not exact zeros"
    if lse is not None:
        ref_l = (torch.logsumexp(s, -1) / LN2).permute(0, 1, 2)  # [B, H, Sq]
        seen = ~empty[:, None, :].expand_as(ref_l)
        assert bool((lse[~seen] == float("inf")).all()), f"{what}: lse of an empty row"
        d = (lse.double()[seen] - ref_l[seen]).abs()
        assert d.numel() == 0 or float(d.max()) <= LSE_TOL, f"{what}: lse error {float(d.max()):.3g}"


@pytest.mark.parametrize("hd", [16, 32, 64])
@pytest.mark.parametrize("band", [1, 2, 7, "wide"])
@pytest.mark.parametrize("Sq,Sk", [(1, 65), (1, 1000), (70, 300), (70, 1000), (256, 65), (256, 300), (256, 1000),
                                   (70, 65), (1, 300)])
def test_band_kernel_matches_fp64(hd, band, Sq, Sk):
    from frankenstein_b200 import _lib
    H = 2
    g = torch.Generator().manual_seed(hd * 1000 + Sq * 7 + Sk + (0 if band == "wide" else band))
    labels = _ring_labels(3, Sq, Sk, 37 if Sk > 65 else 5, g, extreme=True)
    band = 2 ** 32 - 1 if band == "wide" else band
    q, k, v = _operands(3, Sq, Sk, H, hd, g)
    max_chunks = (Sk + 127) // 128
    for nch in sorted({1, min(2, max_chunks), max_chunks}):
        rc, out, lse = _launch_band(q, k, v, H, labels, nch, band)
        assert rc == 0, _lib.lib().fk_last_error()
        _check_band(out, lse, q, k, v, H, labels, band, f"hd {hd} band {band} Sq {Sq} Sk {Sk} chunks {nch}")
    assert _counters_zero()


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_band_kernel_invariants(hd):
    from frankenstein_b200 import _lib, ops
    H, Sq, Sk = 2, 256, 1000
    g = torch.Generator().manual_seed(hd)
    labels = _ring_labels(3, Sq, Sk, 37, g, extreme=True)
    q, k, v = _operands(3, Sq, Sk, H, hd, g)
    max_chunks = (Sk + 127) // 128
    # labels away from the sentinels: a finite band wider than every span between real labels
    plain = _ring_labels(3, Sq, Sk, 37, g)
    real_q, real_k = plain[0][plain[0] != NO_LABEL].long(), plain[1][plain[1] != HI].long()
    span = int(max(real_q.max(), real_k.max()) - min(real_q.min(), real_k.min()))
    for nch in (1, 2, max_chunks):
        # a band wider than every span: bit for bit the unbanded entry point at the same chunk count
        _, a, la = _launch_band(q, k, v, H, plain, nch, None)
        for wide in (span + 1, 2 ** 32, 2 ** 62):
            _, b_, lb = _launch_band(q, k, v, H, plain, nch, wide)
            assert torch.equal(a.view(torch.int16), b_.view(torch.int16)) and torch.equal(la, lb), (nch, wide)
        # keys outside the band of every query of a row: overwriting them with +-3e38 changes no output bit
        for band in (1, 7):
            _, ref, lref = _launch_band(q, k, v, H, labels, nch, band)
            dead = ~_visible(*labels, band).any(1)                # [B, Sk]
            k2, v2 = k.clone(), v.clone()
            big = torch.where(torch.rand(k.shape, generator=g) < 0.5, -3.0e38, 3.0e38).to(torch.bfloat16).cuda()
            k2[dead], v2[dead] = big[dead], big.flip(-1)[dead]
            _, got, lgot = _launch_band(q, k2, v2, H, labels, nch, band)
            assert torch.equal(ref.view(torch.int16), got.view(torch.int16)) and torch.equal(lref, lgot), (nch, band)
            empty = ~_visible(*labels, band).any(-1)
            assert bool((got[empty] == 0).all())
    # a bad band is rejected before the launch: nothing written, counters untouched
    for bad in (0, -1, -2 ** 63):
        before = _lib.launch_count()
        rc, out, lse = _launch_band(q, k, v, H, labels, 2, bad)
        # (the two launches are the label ranges of the mask _launch_band builds)
        assert rc != 0 and b"band" in _lib.lib().fk_last_error() and _lib.launch_count() == before + 2
        assert bool((out == 0).all()) and bool((lse == 0).all())
    assert _counters_zero()
    # ops.attention_kv routes a banded mask to the banded entry; attention_qkv refuses it
    m = ops.LabelMask(*labels, band=7)
    out = ops.attention_kv(q, k, v, H, m)
    _, ref, _ = _launch_band(q, k, v, H, labels, ops.lib().fk_attn_kv_chunks(3, H, Sq, Sk, 0), 7, lse=False)
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))
    qkv = torch.zeros(1, 64, 3 * H * hd, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(ops.FkError, match="banded"):
        ops.attention_qkv(qkv, H, mask=ops.LabelMask(torch.zeros(1, 64, dtype=torch.int32, device="cuda"), band=2))


# ------------------------------------------------------------------------------------------------
# ring bookkeeping kernel
# ------------------------------------------------------------------------------------------------
def _ring_call(len_in, n_new, E, cap, keys, inv, counts=None):
    from frankenstein_b200 import ops
    len_out = torch.full_like(len_in, -7)
    cnt = None if counts is None else torch.tensor(counts, dtype=torch.int32).cuda()
    return ops.stream_ring_positions(len_in, len_out, n_new, E, cap, keys, inv, cnt), len_out


@pytest.mark.parametrize("B,n_new,E,cap", [(5, 256, 256, 8192), (4, 48, 16, 256), (3, 100, 37, 740)])
def test_ring_positions_match_torch(B, n_new, E, cap):
    from frankenstein_b200 import ops
    from frankenstein_b200.brainformer import rope_inv_freq
    g = torch.Generator().manual_seed(B * n_new)
    inv = rope_inv_freq(32, 10000.0).cuda()
    kid = torch.full((B, cap), HI, dtype=torch.int32).cuda()
    nt = (cap + 63) // 64
    keys = ops.LabelMask.from_ranges(None, kid, None, None, torch.full((B, nt), HI, dtype=torch.int32).cuda(),
                                     torch.full((B, nt), HI, dtype=torch.int32).cuda())
    ref_kid = torch.full((B, cap), HI, dtype=torch.int64)
    lens = torch.zeros(B, dtype=torch.int64)
    lens[-1] = 2 ** 33 + 5                                   # far past int32 tokens (patch index still inside int32)
    for step in range(2 + 3 * cap // n_new):                 # count 0 and full counts, across several wraps
        counts = torch.randint(0, n_new + 1, (B,), generator=g)
        counts[step % B] = 0
        counts[(step + 1) % B] = n_new
        (qid, qmin, qmax, rows, rope), len_out = _ring_call(lens.cuda(), n_new, E, cap, keys, inv, counts.tolist())
        i = torch.arange(n_new)[None]
        p = lens[:, None] + i
        live = i < counts[:, None]
        ref_q = torch.where(live, p // E, NO_LABEL)
        assert torch.equal(qid.cpu().long(), ref_q)
        assert torch.equal(rows.cpu(), torch.where(live, torch.arange(B)[:, None] * cap + p % cap, B * cap).reshape(-1))
        m = ops.LabelMask(qid)
        assert torch.equal(m.qmin, qmin) and torch.equal(m.qmax, qmax)
        for b in range(B):
            pb = p[b, :counts[b]]
            ref_kid[b, pb % cap] = pb // E
        assert torch.equal(kid.cpu().long(), ref_kid), f"step {step}: ring key labels"
        r = ops.LabelMask(kid)
        assert torch.equal(r.qmin, keys.kmin) and torch.equal(r.qmax, keys.kmax), f"step {step}: key tile ranges"
        assert torch.equal(len_out.cpu(), lens + counts)
        ang = torch.where(live, p, 0).reshape(-1, 1).double() * inv.cpu().double()[None]
        ref_rope = torch.stack([torch.cos(ang), torch.sin(ang)], -1)
        assert float((rope.cpu().double() - ref_rope).abs().max()) <= 1e-6
        lens = lens + counts
    # RoPE rows at positions 0, a window, 2^20 and 2^30 within 1e-6 of fp64
    for P in (0, 4096, 2 ** 20, 2 ** 30):
        (_, _, _, _, rope), _ = _ring_call(torch.full((B,), P, dtype=torch.int64).cuda(), n_new, E, cap, keys, inv)
        ang = (P + torch.arange(n_new)).double()[:, None] * inv.cpu().double()[None]
        ref_rope = torch.stack([torch.cos(ang), torch.sin(ang)], -1)
        assert float((rope.view(B, n_new, -1, 2)[0].cpu().double() - ref_rope).abs().max()) <= 1e-6, P


# ------------------------------------------------------------------------------------------------
# models against the fp32 oracle with a dense banded block-causal mask
# ------------------------------------------------------------------------------------------------
def _oracle_encoder(enc, x, first_patch=0):
    """fp32 oracle encoder over the patches of x [1, n * p, E], which are the recording's patches first_patch ...: every
    layer banded block-causal (W patches), RoPE at the absolute positions with a cache built in fp64 and cast."""
    from oracle import brainformer_ref as o
    cfg = enc.config
    sd = {kk: vv.detach().float() for kk, vv in enc.state_dict().items()}
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    xp = o.to_patches(x.float(), p)
    n_tok = xp.shape[1]
    h = torch.nn.functional.linear(xp, sd["transformer.emb.weight"], sd["transformer.emb.bias"])
    h = h + sd["space_embedding"].repeat(1, n_tok // E, 1)
    lab = torch.arange(n_tok, device=x.device) // E
    mask = (lab[None, :] <= lab[:, None]) & (lab[:, None] - lab[None, :] < W)
    pos = (first_patch * E + torch.arange(n_tok)).double()
    ang = pos[:, None] * (1.0 / (cfg.rope_theta ** (torch.arange(0, cfg.head_dim, 2).float() / cfg.head_dim))).double()
    rope = torch.polar(torch.ones_like(ang), ang).to(torch.complex64).to(x.device)
    for i in range(len(enc.transformer.h)):
        h = o.block(sd, f"transformer.h.{i}", h, cfg.n_heads, mask, rope)
    return torch.nn.functional.layer_norm(h, (h.shape[-1],), sd["transformer.ln_f.weight"], sd["transformer.ln_f.bias"], 1e-5)


def _oracle_perceiver(model, ctx):
    """fp32 oracle perceiver over the context tokens ctx [1, S, dim]."""
    from oracle import brainformer_ref as o
    sd = {kk: vv.detach().float() for kk, vv in model.state_dict().items()}
    cfg = model.config
    h = sd["learnable_queries"]
    rope = o.rope_cache(cfg.head_dim, cfg.n_output_tokens, cfg.rope_theta, ctx.device)
    for i in range(len(model.perceiver.h)):
        pre = f"perceiver.h.{i}"
        h = h + o.cross_attention(sd, f"{pre}.cross_attn", o._norm(sd, f"{pre}.ln_1", h, False), ctx, cfg.n_heads)
        h = h + o.mlp(sd, f"{pre}.mlp", o._norm(sd, f"{pre}.ln_2", h, False))
        h = o.block(sd, f"{pre}.sa_block", h, cfg.n_heads, None, rope)
    return torch.nn.functional.linear(o._norm(sd, "perceiver.ln_f", h, False), sd["perceiver.to_motion.weight"],
                                      sd["perceiver.to_motion.bias"])


def _steps(W, n_patches, seed):
    """patch counts of one session's steps: ones and multi-patch steps of at most W, summing to n_patches"""
    rng = random.Random(seed)
    out, t = [], 0
    while t < n_patches:
        n = min(rng.choice([1, 1, 2, 3, W]), n_patches - t)
        out.append(n)
        t += n
    return out


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_encoder_sliding_matches_oracle(hd):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(hd)
    enc = bf.Encoder(bf.MAEConfig(**_enc_cfg(hd))).cuda()
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    n_pat = 5 * W + 3
    x = torch.randn(1, n_pat * p, E).cuda()
    with torch.no_grad():
        ref = _oracle_encoder(enc, x)[0]
    s = enc.stream(1, sliding=True)
    t = 0
    for i, n in enumerate(_steps(W, n_pat, hd)):
        with pytest.MonkeyPatch.context() as m:
            _no_dense_attention(m)
            y = s.step(x[:, t * p:(t + n) * p])
        rel_close(y[0], ref[t * E:(t + n) * E], what=f"step {i} (patches {t} .. {t + n - 1}) vs oracle")
        if t + n <= W:
            with torch.no_grad():
                off = enc(x[:, :(t + n) * p])[0, -n * E:]
            rel_close(y[0], off, what=f"step {i} vs Encoder.forward inside the first window")
        t += n
        assert s.lengths == [t * E]
    assert _counters_zero()


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_brainformer_sliding_matches_oracle(hd):
    model = _brainformer(hd, seed=5 + hd)
    enc = model.encoder
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    n_pat = 5 * W + 2
    x = torch.randn(1, n_pat * p, E).cuda()
    with torch.no_grad():
        ctx = _oracle_encoder(enc, x)
    s = model.stream(1, sliding=True)
    t = 0
    for i, n in enumerate(_steps(W, n_pat, 100 + hd)):
        pred = s.step(x[:, t * p:(t + n) * p])
        t += n
        lo = max(0, t - W) * E
        with torch.no_grad():
            ref = _oracle_perceiver(model, ctx[:, lo:t * E])
        rel_close(pred[0], ref[0], what=f"step {i} pred vs oracle perceiver over the last W patches")
        if t <= W:
            with torch.no_grad():
                _, off = model(x[:, :t * p])
            rel_close(pred[0], off[0], what=f"step {i} pred vs BrainFormer.forward")
    assert _counters_zero()


def test_encoder_sliding_cfg2():
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(2)
    enc = bf.Encoder(bf.MAEConfig(**CFG2)).cuda()
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    L = len(enc.transformer.h)
    n_pat = 3 * W
    x = torch.randn(2, n_pat * p, E).cuda()
    s = enc.stream(2, sliding=True)
    t = 0
    for i, n in enumerate(_steps(W, n_pat, 7)):
        y = s.step(x[:, t * p:(t + n) * p])
        if i % 4 == 1 or t + n == n_pat:
            # the oracle over the receptive field: L layers of W patches reach back L (W - 1) patches
            s0 = max(0, t - L * (W - 1))
            for b in range(2):
                with torch.no_grad():
                    ref = _oracle_encoder(enc, x[b:b + 1, s0 * p:(t + n) * p], first_patch=s0)[0, -n * E:]
                rel_close(y[b], ref, what=f"cfg-2 step {i} row {b}")
        t += n
    assert s.lengths == [n_pat * E] * 2
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# sessions
# ------------------------------------------------------------------------------------------------
def _schedule(B, W, n_steps, seed, max_n=3):
    """[(resets, counts)]: counts 0 .. max_n patches; resets (some long after the ring wrapped)"""
    rng = random.Random(seed)
    out = []
    for i in range(n_steps):
        resets = [r for r in range(B) if rng.random() < 0.04]
        counts = [rng.choice([0, 1, 1, 2, max_n]) for _ in range(B)]
        out.append((resets, counts))
    out[n_steps // 2] = ([1], out[n_steps // 2][1])
    return out


def _drive(stream, enc, sched, seeds, filler="zero", width=3):
    """feed the schedule, each row its session's next counts[r] patches then filler (row r's sessions drawn from seed
    seeds[r]); returns the per-step outputs and, per step and row, (session id, session bins fed so far)"""
    p, E = enc.patch_size, enc.n_electrodes
    gs = [torch.Generator().manual_seed(sd) for sd in seeds]
    gf = torch.Generator().manual_seed(999)
    B = len(sched[0][1])
    n_max = len(sched) * width + 1                  # (fixed per schedule length: each draw advances the row's generator)
    sess = [torch.randn(n_max * p, E, generator=gs[r]).cuda() for r in range(B)]
    fed, sid = [0] * B, [0] * B
    outs, hist = [], []
    for i, (resets, counts) in enumerate(sched):
        if resets:
            stream.reset(resets)
            for r in resets:
                sess[r], fed[r], sid[r] = torch.randn(n_max * p, E, generator=gs[r]).cuda(), 0, sid[r] + 1
        x = _fill((B, width * p, E), filler, gf).cuda()
        for r in range(B):
            x[r, :counts[r] * p] = sess[r][fed[r] * p:(fed[r] + counts[r]) * p]
        out = stream.step(x, counts)
        for r in range(B):
            fed[r] += counts[r]
        outs.append(out.clone())
        hist.append([(sid[r], sess[r][:fed[r] * p]) for r in range(B)])
    return outs, hist


def test_encoder_sliding_sessions():
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(9)
    enc = bf.Encoder(bf.MAEConfig(**_enc_cfg(32))).cuda()
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    B = 4
    sched = _schedule(B, W, 60, seed=1)
    s = enc.stream(B, sliding=True)
    outs, hist = _drive(s, enc, sched, [20, 21, 22, 23])
    assert s.lengths == [h[1].shape[0] // p * E for h in hist[-1]]
    assert max(s.lengths) > 4 * W * E                          # some sessions ran past several windows
    # every row against its own session's oracle
    refs = {}
    for i, (resets, counts) in enumerate(sched):
        for r in range(B):
            n = counts[r] * E
            assert bool((outs[i][r, n:] == 0).all()), f"step {i} row {r}: slots past the count are not zero"
            if n == 0:
                continue
            sid, bins = hist[i][r]
            key = (r, sid)
            if key not in refs:                                # the oracle of the session's final bins covers every step
                last = [h[r][1] for h in hist if h[r][0] == sid][-1]
                with torch.no_grad():
                    refs[key] = _oracle_encoder(enc, last[None])[0]
            t = bins.shape[0] // p
            rel_close(outs[i][r, :n], refs[key][(t - counts[r]) * E:t * E], what=f"step {i} row {r} vs oracle")
    # a row's bits do not depend on the other rows' data, counts or resets
    sched2 = [([r for r in rs if r == 2] + ([0] if i % 7 == 3 else []),
               [c[2] if r == 2 else (i + r) % 4 for r in range(B)]) for i, (rs, c) in enumerate(sched)]
    s2 = enc.stream(B, sliding=True)
    outs2, _ = _drive(s2, enc, sched2, [30, 31, 22, 33])
    for i in range(len(sched)):
        assert torch.equal(outs[i][2], outs2[i][2]), f"step {i}: row 2 depends on the other rows"
    # a row reset after its ring wrapped is bit-identical to a fresh sliding stream fed the same bins
    k = len(sched) // 2
    assert 1 in sched[k][0] and hist[k - 1][1][1].shape[0] > 2 * W * p
    end = next((j for j in range(k + 1, len(sched)) if 1 in sched[j][0]), len(sched))
    bins = hist[end - 1][1][1]
    s4 = enc.stream(B, sliding=True)
    t = 0
    for j in range(k, end):
        c = sched[j][1][1]
        x = torch.zeros(B, 3 * p, E, device="cuda")
        x[1, :c * p] = bins[t * p:(t + c) * p]
        y = s4.step(x, [c if r == 1 else 0 for r in range(B)])
        assert torch.equal(y[1], outs[j][1]), f"step {j}: the reset row differs from a fresh stream"
        t += c
    assert _counters_zero()


@pytest.mark.parametrize("filler", ["nan", "huge"])
def test_sliding_filler_never_matters(filler):
    model = _brainformer(32, seed=4)
    enc = model.encoder
    W = enc.n_patches_per_channel
    sched = _schedule(3, W, 30, seed=5)
    a = model.stream(3, sliding=True)
    b = model.stream(3, sliding=True)
    oa, _ = _drive(a, enc, sched, [6, 7, 8])
    ob, _ = _drive(b, enc, sched, [6, 7, 8], filler=filler)
    for i, (x, y) in enumerate(zip(oa, ob)):
        assert torch.equal(x, y), f"step {i}: {filler} filler changed the prediction"
    for c in b.encoder_stream.caches + b.kv:
        assert bool(torch.isfinite(c).all())


def test_sliding_rejections_change_nothing():
    from frankenstein_b200 import ops
    model = _brainformer(16, seed=8)
    enc = model.encoder
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    s = model.stream(3, sliding=True)
    es = s.encoder_stream
    x = torch.randn(3, 2 * W * p, E).cuda()
    for _ in range(3):
        s.step(x[:, :W * p])
    s.step(x[:, :p], [1, 0, 1])

    def state():
        torch.cuda.synchronize()
        return ([t.clone() for t in es.caches + s.kv + [es._keys.kid, es._keys.kmin, es._keys.kmax]],
                es._len_dev.clone(), es._cur, list(es.lengths))
    before = state()
    for bad in ((x, None), (x[:, :(W + 1) * p], [W + 1, 0, 0]), (x[:, :p], [1, 1]), (x[:, :p], [0, 2, 0]),
                (x[:, :p + 1], None)):
        with pytest.raises(ops.FkError):
            s.step(*bad)
    for bad in ([3], [0, 0], [-1]):
        with pytest.raises(ops.FkError):
            s.reset(bad)
    after = state()
    assert all(torch.equal(u, v) for u, v in zip(before[0], after[0]))
    assert torch.equal(before[1], after[1]) and before[2:] == after[2:]
    assert es.lengths == [(3 * W + 1) * E, 3 * W * E, (3 * W + 1) * E]
    # a reset row's key labels are invalid again
    s.reset([1])
    assert bool((es._keys.kid[1] == HI).all()) and bool((es._keys.kmin[1] == HI).all())
    assert bool((es._keys.kid[0] != HI).any())
    assert _counters_zero()


def test_sliding_step_cost_is_constant():
    """the device launch list of a step is the same at patch 1 and at patch 5 W"""
    from torch.profiler import ProfilerActivity, profile
    model = _brainformer(32, seed=12)
    enc = model.encoder
    p, E, W = enc.patch_size, enc.n_electrodes, enc.n_patches_per_channel
    x = torch.randn(2, p, E).cuda()
    s = model.stream(2, sliding=True)

    def launches():
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            s.step(x)
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    s.step(x)
    first = launches()                                         # patch 1 (the second patch; the first warms the caches)
    while s.lengths[0] < (5 * W - 1) * E:
        s.step(x)
    late = launches()
    assert s.lengths[0] == 5 * W * E
    assert first == late and any("stream_ring_positions" in n for n in first)
    assert _counters_zero()
