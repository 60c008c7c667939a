"""Streaming Brainformer inference: the split-key attention of a step against a key / value cache (fk_attn_forward_kv_tc,
ops.attention_kv) against a float64 reference computed from the kernel's exact bf16 operands, and Encoder.stream /
BrainFormer.stream against the offline forward passes and the fp32 oracle.

Kernel checks are per row: max |error| of a row <= OUT_TOL * max |v| of that (trial, head); rows that see no key are exact
zeros.  Model checks are relative Frobenius errors (bf16 activations, rtol 2e-2).
"""
import pytest
import torch

from tests.test_attention_masks_gpu import OUT_TOL

pytestmark = pytest.mark.gpu

RTOL = 2e-2
E_LABEL = 37                    # tokens per label block of the kernel tests (not a divisor of the 128-key tiles)


def rel_close(a, b, rtol=RTOL, what=""):
    a, b = a.double().cpu(), b.double().cpu()
    err = (a - b).norm().item()
    ref = b.norm().item() + 1e-12
    assert err <= rtol * ref, f"{what}: relative error {err / ref:.4g}"


def _counters_zero():
    from frankenstein_b200 import _lib
    torch.cuda.synchronize()
    return all(int(t.abs().sum()) == 0 for t in _lib._counter_sets.values())


def _no_dense_attention(m):
    """any dense mask or library SDPA on the stream path raises"""
    from frankenstein_b200 import brainformer as bf
    from frankenstein_b200 import ops

    def refuse(*a, **k):
        raise AssertionError("dense mask / library SDPA used on the stream path")
    m.setattr(ops.LabelMask, "dense", refuse)
    m.setattr(bf.F, "scaled_dot_product_attention", refuse)


# ------------------------------------------------------------------------------------------------
# kernel
# ------------------------------------------------------------------------------------------------
def _labels(kind, B, Sq, Sk, g):
    """(qid [B, Sq], kid [B, Sk]) int32 CUDA tensors, or None.  'causal': block-causal labels of a step whose queries are
    the last Sq of Sk positions (Sq > Sk: the first queries see nothing); 'empty_rows': the same with scattered queries
    labelled below every key."""
    if kind == "none":
        return None
    kid = (torch.arange(Sk) // E_LABEL).expand(B, Sk).clone()
    qid = ((torch.arange(Sq) + Sk - Sq).div(E_LABEL, rounding_mode="floor")).expand(B, Sq).clone()
    if kind == "empty_rows":
        qid[torch.rand(B, Sq, generator=g) < 0.1] = -1
    return qid.to(torch.int32).cuda(), kid.to(torch.int32).cuda()


def _reference(q, k, v, labels, scale):
    """float64 softmax(q k^T scale + mask) v from the bf16 operands q [B, Sq, H, hd], k / v [B, Sk, H, hd]."""
    qd, kd, vd = q.double(), k.double(), v.double()
    s = torch.einsum("bqhd,bkhd->bhqk", qd, kd) * scale
    if labels is not None:
        qid, kid = labels
        vis = (kid[:, None, None, :] <= qid[:, None, :, None])
        s = s.masked_fill(~vis, float("-inf"))
    p = torch.softmax(s, dim=-1).nan_to_num(0.0)            # rows without a visible key -> zeros
    return torch.einsum("bhqk,bkhd->bqhd", p, vd)


def _check(out, ref, v, labels, what):
    """out [B, Sq, H*hd] bf16 against ref [B, Sq, H, hd] float64, per row."""
    B, Sq, H, hd = ref.shape
    o = out.view(B, Sq, H, hd).double()
    vmax = v.double().abs().amax(dim=(1, 3))                 # [B, H]
    err = (o - ref).abs().amax(dim=3)                        # [B, Sq, H]
    assert bool((err <= OUT_TOL * vmax[:, None, :] + 1e-6).all()), f"{what}: max row error {float((err / vmax[:, None, :]).max()):.3g}"
    if labels is not None:
        qid, kid = labels
        empty = qid < kid.amin(dim=1, keepdim=True)          # [B, Sq]: sees no key
        assert bool((o[empty] == 0).all()), f"{what}: rows that see no key are not exact zeros"


def _operands(B, Sq, Sk, H, hd, seed, amp=1.5):
    g = torch.Generator().manual_seed(seed)
    q = (torch.randn(B, Sq, H * hd, generator=g) * amp).to(torch.bfloat16).cuda()
    k = (torch.randn(B, Sk, H * hd, generator=g) * amp).to(torch.bfloat16).cuda()
    v = torch.randn(B, Sk, H * hd, generator=g).to(torch.bfloat16).cuda()
    return q, k, v, g


def _launch(q, k, v, H, labels, n_chunks, head_dim=None, Sq=None, Sk=None, k_ts=None):
    """raw fk_attn_forward_kv_tc with an explicit chunk count; returns (rc, out)."""
    from frankenstein_b200 import _lib, ops
    from frankenstein_b200._lib import counters, lib, ptr, stream
    B = q.shape[0]
    Sq = q.shape[1] if Sq is None else Sq
    Sk = k.shape[1] if Sk is None else Sk
    hd = q.shape[2] // H if head_dim is None else head_dim
    m = None if labels is None else ops.LabelMask(*labels)
    out = torch.zeros(B, max(Sq, 1), q.shape[2], device=q.device, dtype=torch.bfloat16)
    nc = max(n_chunks, 1)
    part_o = torch.empty(B, H, nc, max(Sq, 1), max(hd, 1), device=q.device, dtype=torch.float32)
    part_ml = torch.empty(B, H, nc, max(Sq, 1), 2, device=q.device, dtype=torch.float32)
    margs = (ptr(m.qid) if m else 0, ptr(m.kid) if m else 0, ptr(m.qmin) if m else 0, ptr(m.qmax) if m else 0,
             ptr(m.kmin) if m else 0, ptr(m.kmax) if m else 0)
    rc = lib().fk_attn_forward_kv_tc(ptr(q), ptr(k), ptr(v), ptr(out), None, B, H, Sq, Sk, hd, q.stride(0), q.stride(1),
                                     k.stride(0), k.stride(1) if k_ts is None else k_ts, v.stride(0), v.stride(1),
                                     out.stride(0), out.stride(1), *margs, float(hd ** -0.5) if hd > 0 else 1.0,
                                     ptr(part_o), ptr(part_ml), n_chunks, counters(_lib.CTR_ATTN_FWD), stream())
    return rc, out


@pytest.mark.parametrize("hd", [16, 32, 64])
@pytest.mark.parametrize("Sq,Sk", [(1, 1), (70, 300), (256, 4096), (700, 6144), (300, 70), (256, 1), (1, 6144)])
@pytest.mark.parametrize("kind", ["none", "causal", "empty_rows"])
def test_attention_kv_matches_fp64(hd, Sq, Sk, kind):
    from frankenstein_b200 import ops
    H = 2
    q, k, v, g = _operands(1, Sq, Sk, H, hd, seed=Sq * 7 + Sk + hd)
    labels = _labels(kind, 1, Sq, Sk, g)
    mask = None if labels is None else ops.LabelMask(*labels)
    with torch.no_grad():
        out = ops.attention_kv(q, k, v, H, mask)
    ref = _reference(q.view(1, Sq, H, hd), k.view(1, Sk, H, hd), v.view(1, Sk, H, hd), labels, hd ** -0.5)
    _check(out, ref, v.view(1, Sk, H, hd), labels, f"hd {hd} Sq {Sq} Sk {Sk} {kind}")
    assert _counters_zero()


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_attention_kv_chunk_counts(hd):
    """every chunk count from 1 (the unsplit kernel) to one chunk per key tile gives the reference result; counts that do
    not divide the tiles leave trailing chunks empty"""
    H, Sq, Sk = 3, 300, 2000                                  # 16 key tiles, ragged tail
    q, k, v, g = _operands(2, Sq, Sk, H, hd, seed=hd)
    labels = _labels("empty_rows", 2, Sq, Sk, g)
    ref = _reference(q.view(2, Sq, H, hd), k.view(2, Sk, H, hd), v.view(2, Sk, H, hd), labels, hd ** -0.5)
    for n in (1, 2, 3, 5, 7, 9, 16):
        rc, out = _launch(q, k, v, H, labels, n)
        assert rc == 0, n
        _check(out, ref, v.view(2, Sk, H, hd), labels, f"hd {hd} chunks {n}")
    assert _counters_zero()


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_attention_kv_strided_cache_views(hd):
    """q a slice of a fused q|k|v projection, k / v the first Sk tokens of a longer [B, cap, 2W] cache: read in place"""
    from frankenstein_b200 import ops
    B, H, Sq, Sk, cap = 2, 4, 256, 1500, 4096
    W = H * hd
    g = torch.Generator().manual_seed(5)
    qkv = (torch.randn(B, Sq, 3 * W, generator=g) * 1.5).to(torch.bfloat16).cuda()
    cache = (torch.randn(B, cap, 2 * W, generator=g) * 1.5).to(torch.bfloat16).cuda()
    q, k, v = qkv[..., :W], cache[:, :Sk, :W], cache[:, :Sk, W:]
    labels = _labels("causal", B, Sq, Sk, g)
    with torch.no_grad():
        out = ops.attention_kv(q, k, v, H, ops.LabelMask(*labels))
    ref = _reference(q.reshape(B, Sq, H, hd), k.reshape(B, Sk, H, hd), v.reshape(B, Sk, H, hd), labels, hd ** -0.5)
    _check(out, ref, v.reshape(B, Sk, H, hd), labels, f"strided hd {hd}")
    assert _counters_zero()


def test_attention_kv_deterministic_and_concurrent():
    from frankenstein_b200 import ops
    H, hd = 16, 32
    ins = [_operands(1, 256, 4096, H, hd, seed=s)[:3] for s in (1, 2)]
    with torch.no_grad():
        serial = [ops.attention_kv(*t, H) for t in ins]
        again = [ops.attention_kv(*t, H) for t in ins]
        assert all(torch.equal(a, b) for a, b in zip(serial, again))
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        torch.cuda.synchronize()
        outs = [None, None]
        for _ in range(3):
            with torch.cuda.stream(s1):
                outs[0] = ops.attention_kv(*ins[0], H)
            with torch.cuda.stream(s2):
                outs[1] = ops.attention_kv(*ins[1], H)
        torch.cuda.synchronize()
    assert torch.equal(outs[0], serial[0]) and torch.equal(outs[1], serial[1])
    assert _counters_zero()


def test_attention_kv_rejections():
    from frankenstein_b200 import ops
    H = 2
    for hd in (48, 128):
        q, k, v, _ = _operands(1, 64, 256, H, hd, seed=hd)
        with torch.no_grad(), pytest.raises(ops.FkError):
            ops.attention_kv(q, k, v, H)
        rc, _ = _launch(q, k, v, H, None, 1, head_dim=hd)
        assert rc != 0
    q, k, v, g = _operands(1, 64, 256, H, 32, seed=3)
    assert _launch(q, k, v, H, None, 1, Sq=0)[0] != 0
    assert _launch(q, k, v, H, None, 1, Sk=0)[0] != 0
    assert _launch(q, k, v, H, None, 1, k_ts=4)[0] != 0               # token stride breaks 16-byte alignment
    assert _launch(q, k, v, H, None, 3)[0] != 0                       # 3 chunks of 2 key tiles
    assert _launch(q, k, v, H, None, 0)[0] != 0
    with pytest.raises(ops.FkError):
        ops.attention_kv(q, k[:, :, :32], v, H)
    qg = q.float().requires_grad_(True).to(torch.bfloat16)
    with pytest.raises(ops.FkError, match="inference"):
        ops.attention_kv(qg, k, v, H)
    torch.cuda.synchronize()
    assert _counters_zero()
    rc, out = _launch(q, k, v, H, None, 2)                            # the next valid launch is correct
    assert rc == 0
    ref = _reference(q.view(1, 64, H, 32), k.view(1, 256, H, 32), v.view(1, 256, H, 32), None, 32 ** -0.5)
    _check(out, ref, v.view(1, 256, H, 32), None, "after rejections")
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# Encoder.stream / BrainFormer.stream
# ------------------------------------------------------------------------------------------------
def _enc_cfg(hd, **kw):
    cfg = dict(window_size=64, n_electrodes=16, patch_size=8, dim=128, n_layers=2, head_dim=hd, hidden_dim=256,
               n_heads=128 // hd, n_kv_heads=128 // hd)
    cfg.update(kw)
    return cfg


CFG2 = dict(window_size=512, n_electrodes=256, patch_size=32, dim=512, n_layers=2, head_dim=32, hidden_dim=2048,
            n_heads=16, n_kv_heads=16)


def _run_stream(enc, x, steps, monkeypatch, oracle_at=None):
    """feed x [B, T, E] in steps of the given patch counts; compare every step with the offline forward on the bins so far
    and, at the steps in oracle_at (all when None), with the fp32 oracle.  Returns the list of step outputs."""
    from oracle import brainformer_ref as o
    stream = enc.stream(x.shape[0])
    p, E = enc.patch_size, enc.n_electrodes
    sd = {kk: vv.detach().float() for kk, vv in enc.state_dict().items()}
    cfg = dict(window_size=enc.config.window_size, patch_size=p, n_electrodes=E, head_dim=enc.config.head_dim,
               n_heads=enc.config.n_heads, rope_theta=enc.config.rope_theta)
    outs, done = [], 0
    for i, n in enumerate(steps):
        with monkeypatch.context() as m:
            _no_dense_attention(m)
            y = stream.step(x[:, done * p:(done + n) * p])
        assert not y.requires_grad and y.dtype == torch.float32 and y.shape == (x.shape[0], n * E, enc.config.dim)
        done += n
        assert stream.length == done * E
        with torch.no_grad():
            off = enc(x[:, :done * p])[:, -n * E:]
        rel_close(y, off, what=f"step {i} vs Encoder.forward")
        if oracle_at is None or i in oracle_at:
            with torch.no_grad():
                ref = o.encoder_forward(sd, x[:, :done * p].float(), cfg)[:, -n * E:]
            rel_close(y, ref, what=f"step {i} vs oracle")
        outs.append(y)
    return stream, outs


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_encoder_stream_small(hd, monkeypatch):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(hd)
    enc = bf.Encoder(bf.MAEConfig(**_enc_cfg(hd))).cuda()
    x = torch.randn(2, 64, 16).cuda()
    _run_stream(enc, x, [1] * 8, monkeypatch)
    _run_stream(enc, x, [1, 3, 4], monkeypatch)
    assert _counters_zero()


def test_encoder_stream_cfg2(monkeypatch):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(2)
    enc = bf.Encoder(bf.MAEConfig(**CFG2)).cuda()
    x = torch.randn(2, 512, 256).cuda()
    _run_stream(enc, x, [1] * 16, monkeypatch, oracle_at={0, 7, 15})
    _run_stream(enc, x, [1, 3, 12], monkeypatch, oracle_at={2})
    assert _counters_zero()


def test_encoder_stream_capacity_and_state():
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(0)
    enc = bf.Encoder(bf.MAEConfig(**_enc_cfg(32))).cuda()
    x = torch.randn(2, 64, 16).cuda()
    s = enc.stream(2)
    first = [s.step(x[:, i * 8:(i + 1) * 8]) for i in range(3)]
    for bad in (x[:, :12],                      # partial patch
                x[:1, :8],                      # wrong batch size
                x[:, :8, :8],                   # wrong electrode count
                x[:, :48]):                     # 3 + 6 patches > 8
        with pytest.raises(bf.ops.FkError):
            s.step(bad)
        assert s.length == 3 * 16
    rest = s.step(x[:, 24:64])                  # the state is still usable: the remaining 5 patches fill the window
    assert s.length == enc.block_size
    with pytest.raises(bf.ops.FkError):
        s.step(x[:, :8])
    with torch.no_grad():
        rel_close(rest, enc(x)[:, 3 * 16:], what="after rejected steps")
    s.reset()
    assert s.length == 0
    again = [s.step(x[:, i * 8:(i + 1) * 8]) for i in range(3)]
    assert all(torch.equal(a, b) for a, b in zip(first, again))
    assert _counters_zero()


@pytest.mark.parametrize("hd", [16, 64])
def test_brainformer_stream_matches_forward(hd, monkeypatch):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(11)
    per = dict(n_output_tokens=8, output_dim=24, dim=128, n_layers=2, head_dim=16, hidden_dim=256, n_heads=8, n_kv_heads=8)
    model = bf.BrainFormer(bf.Config(encoder=bf.MAEConfig(**_enc_cfg(hd)), **per)).cuda()
    with torch.no_grad():
        model.learnable_queries.normal_()
    x = torch.randn(2, 64, 16).cuda()
    s = model.stream(2)
    done = 0
    for n in (1, 2, 1, 4):
        with monkeypatch.context() as m:
            _no_dense_attention(m)
            pred = s.step(x[:, done * 8:(done + n) * 8])
        done += n
        assert s.length == done * 16 and not pred.requires_grad
        with torch.no_grad():
            _, ref = model(x[:, :done * 8])
        rel_close(pred, ref, what=f"pred after {done} patches")
    assert _counters_zero()
