"""Self-attention at head_dim 16 on the tcgen05 kernels (attention_tc.cu: attn_fwd_tc_kernel<16>,
attn_bwd_tc_kernel<.., 16>, attn_aug_kernel<16>), the 16-wide RoPE (fk_rope, GEMM epilogue 5) and the models built with
head_dim=16: float64 parity under every label-mask family of test_attention_masks_gpu.py, fp32 references on the same
bf16-rounded inputs, and the head-dim-generic oracle (oracle/brainformer_ref.py)."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests.test_attention_masks_gpu import (DQ_ROW_TOL, GRAD_TOL, KINDS, LSE_TOL, OUT_TOL, _rope_fp64, errors,
                                            grad_floors, make_labels, reference, run_ops, visibility)

pytestmark = pytest.mark.gpu

RTOL = 2e-2
HD = 16
SHAPES = [1, 63, 65, 129, 300, 513, 1000]


def close(a, b, rtol=RTOL, what=""):
    a, b = a.float().cpu(), b.float().cpu()
    scale = b.abs().max().item() + 1e-12
    err = (a - b).abs().max().item()
    assert err <= rtol * scale, f"{what}: max err {err:.4g} vs scale {scale:.4g}"


def rel_close(a, b, rtol=RTOL, what="", floor=0.0):
    a, b = a.float().cpu(), b.float().cpu()
    err = (a - b).norm().item()
    ref = max(b.norm().item(), floor) + 1e-12
    assert err <= rtol * ref, f"{what}: relative error {err / ref:.4g}"


def _inputs(B, S, H, seed, amp=1.5):
    g = torch.Generator().manual_seed(seed)
    qkv = (torch.randn(B, S, 3 * H * HD, generator=g) * amp).to(torch.bfloat16).cuda()
    d_o = torch.randn(B, S, H * HD, generator=g).to(torch.bfloat16).cuda()
    return qkv, d_o, g


def check16(qkv, H, labels, d_o, what, rope=None, rope_ref=None):
    """ops.attention_qkv at head_dim 16 against the float64 reference, with the tolerances and exact-zero rules of
    test_attention_masks_gpu.py."""
    B, S, _ = qkv.shape
    sc = HD ** -0.5
    got, (q, k, v) = run_ops(qkv, H, labels, d_o, None, rope)
    vis = visibility(labels, B, S, qkv.device)
    ref = reference(q, k, v, vis, sc, d_o.view(B, S, H, HD))
    if rope_ref is not None:
        ref["dq"], ref["dk"] = rope_ref(ref["dq"]), rope_ref(ref["dk"])
    e = errors(got, ref, v, vis, grad_floors(q, k, v, d_o, sc))
    print(f"ERR {what} " + " ".join(f"{k}={x:.3g}" if isinstance(x, float) else f"{k}={x}" for k, x in e.items()))
    assert e["out"] <= OUT_TOL, f"{what}: out per-row error {e['out']:.4g}"
    assert e["lse"] <= LSE_TOL, f"{what}: lse error {e['lse']:.4g}"
    assert not e["empty_lse"], f"{what}: a row with no visible key has a finite lse"
    assert e["empty_out"] == 0.0, f"{what}: a row with no visible key has a non-zero output"
    for name in ("dq", "dk", "dv"):
        assert e[name] <= GRAD_TOL, f"{what}: {name} relative error {e[name]:.4g}"
    assert e["dq_row"] <= DQ_ROW_TOL, f"{what}: dq per-row error {e['dq_row']:.4g}"
    assert e["empty_dq"] == 0.0, f"{what}: a row with no visible key has a non-zero dq"
    assert e["unseen_dkv"] == 0.0, f"{what}: a key no query sees has a non-zero dk / dv"
    return got


# ------------------------------------------------------------------------------------------------
# float64 parity over the mask families
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("S", SHAPES)
def test_masks_hd16(S, kind):
    B, H = 2, 2
    qkv, d_o, g = _inputs(B, S, H, 1000 * S + KINDS.index(kind) + 16)
    check16(qkv, H, make_labels(kind, B, S, g), d_o, f"hd16 {kind} S={S}")


@pytest.mark.parametrize("B,S,H,kind", [(1, 1, 1, "none"), (2, 33, 2, "block48"), (2, 33, 2, "none"),
                                        (1, 4100, 1, "block64"), (1, 4100, 2, "none")])
def test_hd16_edge_shapes(B, S, H, kind):
    qkv, d_o, g = _inputs(B, S, H, 17 * S + B)
    check16(qkv, H, make_labels(kind, B, S, g), d_o, f"edge {B, S, H} {kind}")


def test_hd16_fully_padded_sample():
    """sample 1 is padding only: no query sees a key -> exact zeros in its output and every gradient, lse = +inf."""
    B, S, H = 2, 200, 2
    qkv, d_o, _ = _inputs(B, S, H, 5)
    pad = torch.zeros(B, S, dtype=torch.bool)
    pad[0, 150:] = True
    pad[1, :] = True
    labels = (torch.where(pad, -1, 0), torch.where(pad, 2 ** 31 - 1, 0))
    got = check16(qkv, H, labels, d_o, "fully padded sample")
    for name in ("out", "dq", "dk", "dv"):
        assert got[name][1].abs().max().item() == 0.0, name
    assert torch.isinf(got["lse"][1]).all() and (got["lse"][1] > 0).all()


def test_hd16_invisible_keys_change_nothing():
    """queries labelled <= 7 cannot see keys labelled > 7: new k / v for those keys leave their out, lse and dq bits."""
    B, S, H = 2, 513, 2
    qkv, d_o, g = _inputs(B, S, H, 91)
    qid = torch.randint(0, 16, (B, (S + 31) // 32), generator=g).repeat_interleave(32, dim=1)[:, :S]
    labels = (qid, torch.randint(0, 16, (B, S), generator=g))
    a, _ = run_ops(qkv, H, labels, d_o)
    pert = qkv.clone().view(B, S, 3, H * HD)
    hidden = (labels[1] > 7).cuda()
    pert[:, :, 1:][hidden] = (torch.randn(int(hidden.sum()), 2, H * HD, generator=g) * 3).to(torch.bfloat16).cuda()
    b_, _ = run_ops(pert.view(B, S, -1), H, labels, d_o)
    sel = (labels[0] <= 7).cuda()
    assert sel.any() and hidden.any()
    assert torch.equal(a["out"][sel], b_["out"][sel])
    assert torch.equal(a["dq"][sel], b_["dq"][sel])
    assert torch.equal(a["lse"].permute(0, 2, 1)[sel], b_["lse"].permute(0, 2, 1)[sel])


# ------------------------------------------------------------------------------------------------
# RoPE: fk_rope, GEMM epilogue 5, and the inverse rotation fused into the backward
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("per_sample", [False, True])
def test_attention_hd16_rope(per_sample):
    """RopeSpec with an offset (rope[-T:]) and with per-sample positions: q / k rotated by fk_rope, dq / dk rotated back
    inside the backward kernels."""
    from frankenstein_b200 import ops
    from frankenstein_b200.brainformer import build_complex_rope_cache
    B, S, H, P = 2, 300, 2, 1024
    qkv, d_o, g = _inputs(B, S, H, 31 + per_sample)
    cache = build_complex_rope_cache(HD, P, 10000)
    table = torch.view_as_real(cache).float().contiguous().cuda()
    if per_sample:
        pos = torch.stack([torch.sort(torch.randperm(P, generator=g)[:S])[0] for _ in range(B)]).cuda()
        spec = ops.RopeSpec(table, pos, 0)
    else:
        spec = ops.RopeSpec.from_complex(cache.cuda(), S, last=True)
        pos = (torch.arange(S, device="cuda") + spec.offset).expand(B, S)
    check16(qkv, H, make_labels("gathered" if per_sample else "block48", B, S, g), d_o, f"rope {per_sample}",
            rope=spec, rope_ref=_rope_fp64(table, pos, inverse=True))


@pytest.mark.parametrize("per_sample", [False, True])
def test_rope16_kernel_forward_and_inverse(per_sample):
    from frankenstein_b200 import ops
    from frankenstein_b200.brainformer import apply_rope, build_complex_rope_cache
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
    close(xd, ref, rtol=1e-2, what="rope16")
    ops._rope_inplace(xd, spec, True)
    close(xd, x, rtol=2e-2, what="rope16 inverse")


@pytest.mark.parametrize("M,per_sample", [(4096, False), (300, False), (4096, True), (300, True)])
def test_gemm_rope16_epilogue(M, per_sample):
    """fused q | k | v projection with epilogue 5 == apply_rope on the q / k heads of a plain GEMM (M = 300 runs the
    single-CTA kernel, M = 4096 the CTA-pair kernel)."""
    from frankenstein_b200 import gemm, ops
    from frankenstein_b200.brainformer import apply_rope, build_complex_rope_cache
    H, dim, S = 8, 256, 100 if M == 300 else 512
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
    close(got, ref, rtol=1e-2, what="epilogue 5")


# ------------------------------------------------------------------------------------------------
# forward regimes, full size, determinism, rejections
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("growth", [0.02, 0.2, 2.0])
def test_attention_hd16_running_max_paths(growth):
    """scores that keep growing along the key axis: below the lazy-rescale slack, above it (deferred O rescale) and above
    what the optimistic sweep absorbs (tile redone with its true maximum)."""
    from frankenstein_b200 import ops
    B, S, H = 1, 1024, 2
    g = torch.Generator().manual_seed(7)
    u = torch.nn.functional.normalize(torch.randn(HD, generator=g), dim=0)
    q = torch.randn(B, S, H, HD, generator=g) * 0.3 + u * math.sqrt(float(HD)) * math.log(2.0)
    k = torch.randn(B, S, H, HD, generator=g) * 0.3 + u * (growth * torch.arange(S).float())[None, :, None, None]
    v = torch.randn(B, S, H, HD, generator=g)
    qkv = torch.stack([q, k, v], dim=2).reshape(B, S, 3 * H * HD).cuda().to(torch.bfloat16)
    out = ops.attention_qkv(qkv.clone(), H, None, None)
    qf, kf, vf = qkv.float().view(B, S, 3, H, HD).unbind(2)
    ref = F.scaled_dot_product_attention(qf.transpose(1, 2), kf.transpose(1, 2), vf.transpose(1, 2)).transpose(1, 2)
    assert torch.isfinite(out.float()).all()
    close(out.reshape(B, S, H, HD), ref, what=f"running-max path, growth {growth}")


def test_attention_hd16_full_size_properties():
    """S = 4096, 32 heads x 16, block-causal with 256 electrodes: exact block causality (outputs and gradients of earlier
    time steps bit-identical when later keys / values change, zero gradient to later tokens), linearity in V, row spot
    check against fp32 softmax."""
    from frankenstein_b200 import ops
    B, S, H, E = 2, 4096, 32, 256
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


def test_attention_hd16_deterministic_and_reentrant():
    """two runs are bit-identical; the same work on two streams at once equals the serial run; the caller-owned counter
    words are back at zero after every launch."""
    B, S, H = 2, 1024, 8
    qkv, d_o, g = _inputs(B, S, H, 3)
    qkv2, d_o2, _ = _inputs(B, S, H, 4)
    labels = make_labels("block48", B, S, g)
    r1, _ = run_ops(qkv, H, labels, d_o)
    assert _counters_zero()
    r1b, _ = run_ops(qkv, H, labels, d_o)
    r2, _ = run_ops(qkv2, H, labels, d_o2)
    for name in ("out", "lse", "dq", "dk", "dv"):
        assert torch.equal(r1[name], r1b[name]), name
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        a1, _ = run_ops(qkv, H, labels, d_o)
    with torch.cuda.stream(s2):
        a2, _ = run_ops(qkv2, H, labels, d_o2)
    torch.cuda.synchronize()
    for name in ("out", "lse", "dq", "dk", "dv"):
        assert torch.equal(a1[name], r1[name]) and torch.equal(a2[name], r2[name]), name
    assert _counters_zero()


@pytest.mark.parametrize("switch,value", [("ATTN_FWD_IMPL", "legacy"), ("ATTN_BWD_IMPL", "legacy"),
                                          ("ATTN_BWD_OPERANDS", "transposed"), ("ATTN_BWD_STATS", "staged")])
def test_cross_check_switch_rejected_at_hd16(switch, value, monkeypatch):
    from frankenstein_b200 import ops
    qkv, _, _ = _inputs(1, 128, 1, 2)
    monkeypatch.setattr(ops, switch, value)
    with pytest.raises(ops.FkError, match=switch):
        ops.attention_qkv(qkv.clone(), 1, None, None)


# ------------------------------------------------------------------------------------------------
# models built with head_dim 16 against the oracle (fp32 on the GPU)
# ------------------------------------------------------------------------------------------------
def _no_dense_attention(m):
    """any dense mask or library SDPA on the model's path raises"""
    from frankenstein_b200 import brainformer as bf
    from frankenstein_b200 import ops

    def refuse(*a, **k):
        raise AssertionError("dense mask / library SDPA used at head_dim 16")
    m.setattr(ops.LabelMask, "dense", refuse)
    m.setattr(bf.F, "scaled_dot_product_attention", refuse)


def _oracle_sd(model):
    return {k: v.detach().clone().requires_grad_(v.is_floating_point()) for k, v in model.state_dict().items()}


def _grads_match(model, sd, rtol=RTOL):
    floor = 1e-4 * max(sd[n].grad.norm().item() for n, p in model.named_parameters() if p.grad is not None)
    n_checked = 0
    for n, p in model.named_parameters():
        if p.grad is None:
            continue
        assert sd[n].grad is not None, n
        rel_close(p.grad, sd[n].grad, rtol=rtol, what=f"grad {n}", floor=floor)
        n_checked += 1
    assert n_checked > 0


_ENC = dict(window_size=64, n_electrodes=16, patch_size=8, dim=128, n_layers=2, head_dim=16, hidden_dim=256,
            n_heads=8, n_kv_heads=8, n_dec_layers=2, decoder_dim=128)


def test_brainformer_hd16_matches_oracle(monkeypatch):
    """Encoder (block-causal LabelMask + RopeSpec -> fused q|k|v GEMM with epilogue 5 + tcgen05 attention at head_dim 16)
    and the perceiver at head_dim 16 (its self-attention Block stays on the few-query kernels)."""
    from frankenstein_b200 import brainformer as bf
    from oracle import brainformer_ref as o
    torch.manual_seed(0)
    per = dict(n_output_tokens=8, output_dim=24, dim=128, n_layers=2, head_dim=16, hidden_dim=256, n_heads=8, n_kv_heads=8)
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


def test_mae_hd16_matches_oracle(monkeypatch):
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


def test_simple_mae_hd16_matches_oracle(monkeypatch):
    """padding masks (sample 1 ends in 12 all-zero tokens) in the encoder (gathered positions) and the decoder."""
    from frankenstein_b200 import simple_mae as sm
    from oracle import brainformer_ref as o
    torch.manual_seed(3)
    ec = dict(block_size=64, patch_size=16, n_layers=2, dim=128, hidden_dim=256, head_dim=16, n_heads=8, n_kv_heads=8,
              rope_theta=10000)
    mc = dict(n_layers=2, dim=128, hidden_dim=256, head_dim=16, n_heads=8, n_kv_heads=8, rope_theta=10000)
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
