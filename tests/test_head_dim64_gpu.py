"""Self-attention at head_dim 64 on the tcgen05 kernels (attention_tc.cu: attn_fwd_tc_kernel<64>, attn_bwd_tc64_kernel,
attn_aug_kernel<64>), the 64-wide RoPE (fk_rope, GEMM epilogue 4) and the models built with head_dim=64, against fp32
references on the same bf16-rounded inputs and the head-dim-generic oracle (oracle/brainformer_ref.py)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

RTOL = 2e-2
HD = 64


def close(a, b, rtol=RTOL, what=""):
    a, b = a.float().cpu(), b.float().cpu()
    scale = b.abs().max().item() + 1e-12
    err = (a - b).abs().max().item()
    assert err <= rtol * scale, f"{what}: max err {err:.4g} vs scale {scale:.4g}"


def rel_close(a, b, rtol=RTOL, what="", floor=0.0):
    """relative Frobenius error (gradients of whole models: a few entries near zero carry no information); `floor`: norm
    below which a gradient is rounding noise in both implementations."""
    a, b = a.float().cpu(), b.float().cpu()
    err = (a - b).norm().item()
    ref = max(b.norm().item(), floor) + 1e-12
    assert err <= rtol * ref, f"{what}: relative error {err / ref:.4g}"


def _labels(kind, B, S, dev, g):
    from frankenstein_b200.ops import LabelMask
    if kind == "none":
        return None
    if kind == "block64":
        return LabelMask.block_causal(B, S, 64, dev)
    if kind == "block48":
        return LabelMask.block_causal(B, S, 48, dev)
    if kind == "gathered":   # sorted random subset of 4*S positions, block = 32 positions (MAE kept tokens)
        ids = torch.stack([torch.sort(torch.randperm(4 * S, generator=g)[:S])[0] for _ in range(B)])
        return LabelMask((ids // 32).to(dev))
    if kind == "padding":
        pad = torch.zeros(B, S, dtype=torch.bool)
        for b in range(B):
            pad[b, max(S - 17 * (b + 1), 0):] = True
        return LabelMask.padding(pad.to(dev))
    raise ValueError(kind)


def _reference(qkv, H, mask, w, rope=None):
    """fp32 SDPA on the bf16-rounded inputs; rows with no visible key are zero (the kernels' convention)."""
    from frankenstein_b200.brainformer import apply_rope
    B, S, _ = qkv.shape
    ref_in = qkv.float().clone().requires_grad_(True)
    q, k, v = ref_in.view(B, S, 3, H, HD).unbind(2)
    if rope is not None:
        q, k = apply_rope(q, rope), apply_rope(k, rope)
    dense = mask.dense() if mask is not None else None
    r = F.scaled_dot_product_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), attn_mask=dense)
    if dense is not None:
        r = torch.where(dense.any(-1, keepdim=True), r, torch.zeros_like(r))
    r = r.transpose(1, 2).reshape(B, S, H * HD)
    (r * w).sum().backward()
    return r.detach(), ref_in.grad


def _run(qkv, H, mask, w, spec=None):
    from frankenstein_b200 import ops
    x = qkv.clone().requires_grad_(True)
    out = ops.attention_qkv(x * 1.0, H, spec, mask)          # x * 1.0: the kernel wants a non-leaf fresh buffer
    (out.float() * w).sum().backward()
    return out.detach(), x.grad


def _inputs(B, S, H, seed, amp=1.5):
    g = torch.Generator().manual_seed(seed)
    dev = torch.device("cuda")
    qkv = (torch.randn(B, S, 3 * H * HD, generator=g) * amp).to(dev).to(torch.bfloat16)
    w = torch.randn(B, S, H * HD, generator=g).to(dev)
    return qkv, w, g


@pytest.mark.parametrize("kind", ["none", "block64", "block48", "gathered", "padding"])
@pytest.mark.parametrize("B,S,H", [(2, 512, 4), (1, 300, 2), (3, 70, 1)])
def test_attention_hd64_fwd_bwd(kind, B, S, H):
    qkv, w, g = _inputs(B, S, H, B * 1000 + S + 64)
    mask = _labels(kind, B, S, qkv.device, g)
    out, grad = _run(qkv, H, mask, w)
    r, rg = _reference(qkv, H, mask, w)
    close(out, r, what=f"hd64 out {kind}")
    close(grad, rg, rtol=3e-2, what=f"hd64 dqkv {kind}")


@pytest.mark.parametrize("B,S,H,kind", [(1, 1, 1, "none"), (2, 33, 2, "block48"), (1, 4100, 1, "block64"), (2, 33, 2, "none")])
def test_attention_hd64_edge_shapes(B, S, H, kind):
    qkv, w, g = _inputs(B, S, H, 17 * S + B)
    mask = _labels(kind, B, S, qkv.device, g)
    out, grad = _run(qkv, H, mask, w)
    r, rg = _reference(qkv, H, mask, w)
    close(out, r, what=f"edge {B, S, H} out")
    close(grad, rg, rtol=3e-2, what=f"edge {B, S, H} dqkv")


def test_attention_hd64_fully_padded_sample():
    """sample 1 is padding only: no query sees a key -> zero output and zero gradient for the whole sample."""
    from frankenstein_b200.ops import LabelMask
    B, S, H = 2, 200, 2
    qkv, w, _ = _inputs(B, S, H, 5)
    pad = torch.zeros(B, S, dtype=torch.bool)
    pad[0, 150:] = True
    pad[1, :] = True
    mask = LabelMask.padding(pad.cuda())
    out, grad = _run(qkv, H, mask, w)
    assert out[1].abs().max().item() == 0.0 and grad[1].abs().max().item() == 0.0
    r, rg = _reference(qkv, H, mask, w)
    close(out, r, what="padded out")
    close(grad, rg, rtol=3e-2, what="padded dqkv")


@pytest.mark.parametrize("per_sample", [False, True])
def test_attention_hd64_rope(per_sample):
    """RopeSpec with an offset (rope[-T:]) and with per-sample positions (MAE gathered tokens): q / k rotated by fk_rope,
    dq / dk rotated back inside the backward kernels."""
    from frankenstein_b200 import ops
    from frankenstein_b200.brainformer import build_complex_rope_cache
    B, S, H, P = 2, 300, 2, 1024
    qkv, w, g = _inputs(B, S, H, 31 + per_sample)
    cache = build_complex_rope_cache(HD, P, 10000)
    mask = _labels("gathered" if per_sample else "block48", B, S, qkv.device, g)
    if per_sample:
        pos = torch.stack([torch.sort(torch.randperm(P, generator=g)[:S])[0] for _ in range(B)])
        spec = ops.RopeSpec(torch.view_as_real(cache).float().cuda(), pos.cuda(), 0)
        ref_rope = cache[pos].cuda()
    else:
        spec = ops.RopeSpec.from_complex(cache.cuda(), S, last=True)
        ref_rope = cache.cuda()
    out, grad = _run(qkv, H, mask, w, spec)
    r, rg = _reference(qkv, H, mask, w, ref_rope)
    close(out, r, what="rope out")
    close(grad, rg, rtol=3e-2, what="rope dqkv")


@pytest.mark.parametrize("per_sample", [False, True])
def test_rope64_kernel_forward_and_inverse(per_sample):
    from frankenstein_b200 import ops
    from frankenstein_b200.brainformer import build_complex_rope_cache, apply_rope
    B, S, H, P = 2, 100, 3, 256
    g = torch.Generator().manual_seed(1)
    cache = build_complex_rope_cache(HD, P, 10000)
    x = torch.randn(B, S, H, HD, generator=g).to(torch.bfloat16)
    if per_sample:
        pos = torch.stack([torch.sort(torch.randperm(P, generator=g)[:S])[0] for _ in range(B)])
        ref = apply_rope(x, cache[pos])
        spec = ops.RopeSpec(torch.view_as_real(cache).float().cuda(), pos.cuda(), 0)
    else:
        ref = apply_rope(x, cache)
        spec = ops.RopeSpec.from_complex(cache.cuda(), S, last=True)
    xd = x.cuda().clone()
    ops._rope_inplace(xd, spec, False)
    close(xd, ref, rtol=1e-2, what="rope64")
    ops._rope_inplace(xd, spec, True)
    close(xd, x, rtol=2e-2, what="rope64 inverse")


@pytest.mark.parametrize("M,per_sample", [(4096, False), (300, False), (4096, True)])
def test_gemm_rope64_epilogue(M, per_sample):
    """fused q | k | v projection with epilogue 4 == apply_rope on the q / k heads of a plain GEMM (M = 300 runs the
    single-CTA kernel, M = 4096 the CTA-pair kernel)."""
    from frankenstein_b200 import gemm, ops
    from frankenstein_b200.brainformer import build_complex_rope_cache, apply_rope
    H, dim, S = 4, 256, 100 if M == 300 else 512
    B = M // S
    g = torch.Generator().manual_seed(M + per_sample)
    cache = build_complex_rope_cache(HD, 1024, 10000)
    x = torch.randn(B, S, dim, generator=g).cuda()
    wq, wk, wv = (torch.randn(H * HD, dim, generator=g).cuda() * dim ** -0.5 for _ in range(3))
    if per_sample:
        pos = torch.stack([torch.sort(torch.randperm(1024, generator=g)[:S])[0] for _ in range(B)])
        spec = ops.RopeSpec(torch.view_as_real(cache).float().cuda(), pos.cuda(), 0)
        rope = cache[pos].cuda()
    else:
        spec = ops.RopeSpec.from_complex(cache.cuda(), S, last=True)
        rope = cache.cuda()
    got = gemm.qkv_rope(x, wq, wk, wv, spec, H).float()
    xb = x.to(torch.bfloat16).float()
    plain = xb @ torch.cat([wq, wk, wv]).to(torch.bfloat16).float().t()
    q, k, v = plain.view(B, S, 3, H, HD).unbind(2)
    ref = torch.stack([apply_rope(q, rope), apply_rope(k, rope), v], dim=2).reshape(B, S, 3 * H * HD)
    close(got, ref, rtol=1e-2, what="epilogue 4")


@pytest.mark.parametrize("growth", [0.02, 0.2, 2.0])
def test_attention_hd64_running_max_paths(growth):
    """scores that keep growing along the key axis: below the lazy-rescale slack, above it (deferred O rescale) and above
    what the optimistic sweep absorbs (tile redone with its true maximum)."""
    from frankenstein_b200 import ops
    B, S, H = 1, 1024, 2
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(7)
    u = torch.nn.functional.normalize(torch.randn(HD, generator=g), dim=0)
    q = torch.randn(B, S, H, HD, generator=g) * 0.3 + u * math.sqrt(float(HD)) * math.log(2.0)
    k = torch.randn(B, S, H, HD, generator=g) * 0.3 + u * (growth * torch.arange(S).float())[None, :, None, None]
    v = torch.randn(B, S, H, HD, generator=g)
    qkv = torch.stack([q, k, v], dim=2).reshape(B, S, 3 * H * HD).to(dev).to(torch.bfloat16)
    out = ops.attention_qkv(qkv.clone(), H, None, None)
    qf, kf, vf = qkv.float().view(B, S, 3, H, HD).unbind(2)
    ref = F.scaled_dot_product_attention(qf.transpose(1, 2), kf.transpose(1, 2), vf.transpose(1, 2)).transpose(1, 2)
    assert torch.isfinite(out.float()).all()
    close(out.reshape(B, S, H, HD), ref, what=f"running-max path, growth {growth}")


def test_attention_hd64_full_size_properties():
    """S = 4096, 8 heads x 64, block-causal with 256 electrodes: exact block causality (outputs and gradients of earlier
    time steps bit-identical when later keys / values change, zero gradient to later tokens), linearity in V, row spot
    check against fp32 softmax."""
    from frankenstein_b200 import ops
    B, S, H, E = 2, 4096, 8, 256
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(11)
    qkv = (torch.randn(B, S, 3 * H * HD, generator=g) * 1.2).to(dev).to(torch.bfloat16)
    mask = ops.LabelMask.block_causal(B, S, E, dev)

    def run(x, w=None):
        xx = x.clone().requires_grad_(True)
        out = ops.attention_qkv(xx * 1.0, H, None, mask)
        if w is None:
            return out.detach(), None
        (out.float() * w).sum().backward()
        return out.detach(), xx.grad.detach()

    w = torch.randn(B, S, H * HD, generator=g).to(dev)
    t0 = 9 * E
    w_early = w.clone(); w_early[:, t0:] = 0
    out_a, grad_a = run(qkv, w_early)
    pert = qkv.clone()
    pert[:, t0:, H * HD:] = (torch.randn(B, S - t0, 2 * H * HD, generator=g) * 1.2).to(dev).to(torch.bfloat16)
    out_b, grad_b = run(pert, w_early)
    assert torch.equal(out_a[:, :t0], out_b[:, :t0]), "outputs of earlier time steps changed with later keys/values"
    assert torch.equal(grad_a[:, :t0], grad_b[:, :t0]), "gradients of earlier tokens changed with later keys/values"
    assert grad_a[:, t0:].abs().max().item() == 0.0, "later tokens received gradient from a loss on earlier time steps"
    v2 = qkv.clone(); v2[..., 2 * H * HD:] = torch.randn(B, S, H * HD, generator=g).to(dev).to(torch.bfloat16)
    vs = qkv.clone(); vs[..., 2 * H * HD:] = (qkv[..., 2 * H * HD:].float() + v2[..., 2 * H * HD:].float()).to(torch.bfloat16)
    o1, _ = run(qkv); o2, _ = run(v2); o3, _ = run(vs)
    close(o3, o1.float() + o2.float(), rtol=2e-2, what="linearity in V")
    q, k, v = qkv.float().view(B, S, 3, H, HD).unbind(2)
    for i in torch.randint(0, S, (64,), generator=g).tolist():
        b, hh = i % B, i % H
        vis = (torch.arange(S, device=dev) // E) <= (i // E)
        sc = (k[b, :, hh] @ q[b, i, hh]) / math.sqrt(float(HD))
        ref = torch.softmax(sc.masked_fill(~vis, float("-inf")), dim=0) @ v[b, :, hh]
        got = o1[b, i].view(H, HD)[hh].float()
        assert (got - ref).abs().max().item() <= 2e-2 * ref.abs().max().item() + 2e-3, f"row {i}"


def _counters_zero():
    from frankenstein_b200 import _lib
    torch.cuda.synchronize()
    return all(int(t.abs().sum()) == 0 for t in _lib._counter_sets.values())


def test_attention_hd64_deterministic_and_reentrant():
    """two runs are bit-identical; the same work on two streams at once equals the serial run; the caller-owned counter
    words are back at zero after every launch."""
    from frankenstein_b200 import ops
    B, S, H = 2, 1024, 4
    qkv, w, g = _inputs(B, S, H, 3)
    qkv2, w2, _ = _inputs(B, S, H, 4)
    mask = _labels("block48", B, S, qkv.device, g)
    o1, g1 = _run(qkv, H, mask, w)
    assert _counters_zero()
    o1b, g1b = _run(qkv, H, mask, w)
    assert torch.equal(o1, o1b) and torch.equal(g1, g1b)
    o2, g2 = _run(qkv2, H, mask, w2)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        r1 = _run(qkv, H, mask, w)
    with torch.cuda.stream(s2):
        r2 = _run(qkv2, H, mask, w2)
    torch.cuda.synchronize()
    assert torch.equal(r1[0], o1) and torch.equal(r1[1], g1)
    assert torch.equal(r2[0], o2) and torch.equal(r2[1], g2)
    assert _counters_zero()


@pytest.mark.parametrize("bad_hd", [48, 128])
def test_attention_rejects_other_head_dims(bad_hd):
    """fk_attn_forward_tc / fk_attn_backward_tc reject head_dim 48 / 128 before launching: FkError, counters untouched,
    and the next valid launch is correct."""
    from frankenstein_b200 import _lib, ops
    from frankenstein_b200._lib import FkError, check, counters, lib, ptr, stream
    B, S, H = 1, 256, 2
    qkv, w, _ = _inputs(B, S, H, 9)
    out = torch.empty(B, S, H * HD, device=qkv.device, dtype=torch.bfloat16)
    lse = torch.empty(B, H, S, device=qkv.device, dtype=torch.float32)
    ts = qkv.stride(1)
    with pytest.raises(FkError):
        check(lib().fk_attn_forward_tc(ptr(qkv), ptr(qkv), ptr(qkv), ptr(out), ptr(lse), B, H, S, bad_hd, qkv.stride(0), ts,
                                       qkv.stride(0), ts, qkv.stride(0), ts, out.stride(0), out.stride(1),
                                       0, 0, 0, 0, 0, 0, 0.125, counters(_lib.CTR_ATTN_FWD), stream()), "bad head_dim")
    aug = torch.empty(B, H, S, 16, device=qkv.device, dtype=torch.bfloat16)
    d = torch.empty_like(qkv)
    with pytest.raises(FkError):
        check(lib().fk_attn_backward_tc(ptr(qkv), ptr(qkv), ptr(qkv), ptr(out), 0, 0, 0, S, ptr(lse), ptr(lse), ptr(aug),
                                        ptr(d), ptr(d), ptr(d), B, H, S, bad_hd, qkv.stride(0), ts, qkv.stride(0), ts,
                                        qkv.stride(0), ts, out.stride(0), out.stride(1), d.stride(0), d.stride(1),
                                        d.stride(0), d.stride(1), d.stride(0), d.stride(1), 0, 0, 0, 0, 0, 0, 0.125,
                                        0, 0, 0, 0, 6, counters(_lib.CTR_ATTN_BWD), stream()), "bad head_dim")
    assert _counters_zero()
    got, grad = _run(qkv, H, None, w)
    r, rg = _reference(qkv, H, None, w)
    close(got, r, what="launch after a rejected one")
    close(grad, rg, rtol=3e-2, what="launch after a rejected one (dqkv)")
    assert _counters_zero()


@pytest.mark.parametrize("switch,value", [("ATTN_FWD_IMPL", "legacy"), ("ATTN_BWD_IMPL", "legacy"),
                                          ("ATTN_BWD_OPERANDS", "transposed"), ("ATTN_BWD_STATS", "staged")])
def test_cross_check_switch_rejected_at_hd64(switch, value, monkeypatch):
    from frankenstein_b200 import ops
    qkv, _, _ = _inputs(1, 128, 1, 2)
    monkeypatch.setattr(ops, switch, value)
    with pytest.raises(ops.FkError, match=switch):
        ops.attention_qkv(qkv.clone(), 1, None, None)


# ------------------------------------------------------------------------------------------------
# models built with head_dim 64 against the oracle (fp32 on the GPU)
# ------------------------------------------------------------------------------------------------
def _no_dense_attention(m):
    """any dense mask or library SDPA on the model's path raises"""
    from frankenstein_b200 import brainformer as bf
    from frankenstein_b200 import ops

    def refuse(*a, **k):
        raise AssertionError("dense mask / library SDPA used at head_dim 64")
    m.setattr(ops.LabelMask, "dense", refuse)
    m.setattr(bf.F, "scaled_dot_product_attention", refuse)


def _oracle_sd(model):
    return {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}


def _grads_match(model, sd, rtol=RTOL):
    # (e.g. the perceiver's self-attention qw / kw see ~1e-8: its few queries are nearly identical at initialisation)
    floor = 1e-4 * max(sd[n].grad.norm().item() for n, p in model.named_parameters() if p.grad is not None)
    n_checked = 0
    for n, p in model.named_parameters():
        if p.grad is None:
            continue
        assert sd[n].grad is not None, n
        rel_close(p.grad, sd[n].grad, rtol=rtol, what=f"grad {n}", floor=floor)
        n_checked += 1
    assert n_checked > 0


_ENC = dict(window_size=64, n_electrodes=16, patch_size=8, dim=128, n_layers=2, head_dim=64, hidden_dim=256,
            n_heads=2, n_kv_heads=2, n_dec_layers=2, decoder_dim=128)


def test_brainformer_hd64_matches_oracle(monkeypatch):
    """Encoder (block-causal LabelMask + RopeSpec -> fused q|k|v GEMM with epilogue 4 + tcgen05 attention) and the
    perceiver (head_dim 64: cross attention and its self-attention Block stay on the few-query kernels)."""
    from frankenstein_b200 import brainformer as bf
    from oracle import brainformer_ref as o
    torch.manual_seed(0)
    per = dict(n_output_tokens=8, output_dim=24, dim=128, n_layers=2, head_dim=64, hidden_dim=256, n_heads=2, n_kv_heads=2)
    full = bf.BrainFormer(bf.Config(encoder=bf.MAEConfig(**_ENC), **per)).cuda()
    x = torch.randn(2, 64, 16).cuda()
    tgt = torch.randn(2, 8, 24).cuda()
    with monkeypatch.context() as m:
        _no_dense_attention(m)
        loss, _ = full(x, tgt)
        loss.backward()
    sd = _oracle_sd(full)
    lr, _ = o.brainformer_forward(sd, x, _ENC, per, tgt)
    lr.backward()
    assert abs(loss.item() - lr.item()) <= RTOL * abs(lr.item()), (loss.item(), lr.item())
    _grads_match(full, sd)


def test_mae_hd64_matches_oracle(monkeypatch):
    from frankenstein_b200 import brainformer as bf
    from oracle import brainformer_ref as o
    torch.manual_seed(1)
    mae = bf.MAE(bf.MAEConfig(**_ENC)).cuda()
    x = torch.randn(2, 64, 16).cuda()
    g = torch.Generator().manual_seed(2)
    order = torch.stack([torch.randperm(128, generator=g) for _ in range(2)])
    masked, unmasked = torch.sort(order[:, :96])[0].cuda(), torch.sort(order[:, 96:])[0].cuda()
    mae.get_masking_indices = lambda r, xx: (masked, unmasked)
    with monkeypatch.context() as m:
        _no_dense_attention(m)
        loss, _ = mae(x)
        loss.backward()
    sd = _oracle_sd(mae)
    lr, _ = o.mae_forward(sd, x, _ENC, masked, unmasked)
    lr.backward()
    assert abs(loss.item() - lr.item()) <= RTOL * abs(lr.item()), (loss.item(), lr.item())
    _grads_match(mae, sd)


def test_simple_mae_hd64_matches_oracle(monkeypatch):
    """padding masks (sample 1 ends in 12 all-zero tokens) in the encoder (gathered positions) and the decoder."""
    from frankenstein_b200 import simple_mae as sm
    from oracle import brainformer_ref as o
    torch.manual_seed(3)
    ec = dict(block_size=64, patch_size=16, n_layers=2, dim=128, hidden_dim=256, head_dim=64, n_heads=2, n_kv_heads=2,
              rope_theta=10000)
    mc = dict(n_layers=2, dim=128, hidden_dim=256, head_dim=64, n_heads=2, n_kv_heads=2, rope_theta=10000)
    model = sm.SimpleMAE(sm.SimpleEncoderConfig(**ec), sm.SimpleMAEConfig(**mc)).cuda()
    x = torch.randn(2, 64, 16)
    x[1, 52:] = 0.0
    x = x.cuda()
    g = torch.Generator().manual_seed(4)
    order = torch.stack([torch.randperm(64, generator=g) for _ in range(2)])
    masked, unmasked = torch.sort(order[:, :32])[0].cuda(), torch.sort(order[:, 32:])[0].cuda()
    model.get_masking_indices = lambda r, xx: (masked, unmasked)
    with monkeypatch.context() as m:
        _no_dense_attention(m)
        loss, _ = model(x, masking_ratio=0.5)
        loss.backward()
    sd = _oracle_sd(model)
    lr, _ = o.simple_mae_forward(sd, x, ec, mc, masked, unmasked)
    lr.backward()
    assert abs(loss.item() - lr.item()) <= RTOL * abs(lr.item()), (loss.item(), lr.item())
    _grads_match(model, sd)
