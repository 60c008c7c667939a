"""GPU parity of the transformer-block kernels and the Brainformer mirror against plain PyTorch fp32 / the CPU
oracle (oracle/brainformer_ref.py).  Tolerance: bf16 compute with fp32 accumulate, rtol 2e-2 (north_star),
measured against the tensor's scale (bf16 outputs carry ~3 significant digits)."""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

RTOL = 2e-2


def close(a, b, rtol=RTOL, what=""):
    a, b = a.float().cpu(), b.float().cpu()
    scale = b.abs().max().item() + 1e-12
    err = (a - b).abs().max().item()
    assert err <= rtol * scale, f"{what}: max err {err:.4g} vs scale {scale:.4g}"


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
            pad[b, S - 17 * (b + 1):] = True
        return LabelMask.padding(pad.to(dev))
    raise ValueError(kind)


@pytest.mark.parametrize("impl", ["tc", "tc-staged", "legacy"])
@pytest.mark.parametrize("kind", ["none", "block64", "block48", "gathered", "padding"])
@pytest.mark.parametrize("B,S,H", [(2, 512, 4), (1, 300, 2), (3, 70, 1)])
def test_attention_fwd_bwd(kind, B, S, H, impl, monkeypatch):
    """tc: tcgen05 kernels, backward row statistics folded into the score MMAs (default); tc-staged: the same kernels reading
    lse / delta themselves (cross-check); legacy: the mma.sync kernels."""
    from frankenstein_b200 import ops
    monkeypatch.setattr(ops, "ATTN_BWD_STATS", "staged" if impl == "tc-staged" else "folded")
    impl = "tc" if impl == "tc-staged" else impl
    monkeypatch.setattr(ops, "ATTN_BWD_IMPL", impl)
    monkeypatch.setattr(ops, "ATTN_FWD_IMPL", impl)
    g = torch.Generator().manual_seed(B * 1000 + S)
    dev = torch.device("cuda")
    qkv = (torch.randn(B, S, 3 * H * 32, generator=g) * 1.5).to(dev).to(torch.bfloat16)
    w = torch.randn(B, S, H * 32, generator=g).to(dev)
    mask = _labels(kind, B, S, dev, g)
    x = qkv.clone().requires_grad_(True)
    out = ops.attention_qkv(x * 1.0, H, None, mask)          # x * 1.0: the kernel wants a non-leaf fresh buffer
    (out.float() * w).sum().backward()
    ref_in = qkv.float().clone().requires_grad_(True)
    q, k, v = ref_in.view(B, S, 3, H, 32).unbind(2)
    dense = mask.dense() if mask is not None else None
    r = F.scaled_dot_product_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2), attn_mask=dense)
    if dense is not None:
        r = torch.where(dense.any(-1, keepdim=True), r, torch.zeros_like(r))
    r = r.transpose(1, 2).reshape(B, S, H * 32)
    (r * w).sum().backward()
    close(out, r, what=f"attention out {kind}")
    close(x.grad, ref_in.grad, rtol=3e-2, what=f"attention dqkv {kind}")


@pytest.mark.parametrize("growth", [0.02, 0.2, 2.0])
def test_attention_forward_running_max_paths(growth):
    """Scores that keep growing along the key axis: per 128-key tile the row maximum rises by less than the lazy-rescale
    slack (growth 0.02), by more than the slack (0.2: deferred O rescale) and by more than the optimistic sweep can absorb
    (2.0: the tile is redone with its true maximum) -- forward values must match fp32 SDPA in every regime."""
    from frankenstein_b200 import ops
    B, S, H = 1, 1024, 2
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(7)
    u = torch.nn.functional.normalize(torch.randn(32, generator=g), dim=0)
    q = torch.randn(B, S, H, 32, generator=g) * 0.3 + u * math.sqrt(32.0) * math.log(2.0)     # q.u*scale ~ ln 2 per unit of k.u
    k = torch.randn(B, S, H, 32, generator=g) * 0.3 + u * (growth * torch.arange(S).float())[None, :, None, None]
    v = torch.randn(B, S, H, 32, generator=g)
    qkv = torch.stack([q, k, v], dim=2).reshape(B, S, 3 * H * 32).to(dev).to(torch.bfloat16)
    out = ops.attention_qkv(qkv.clone(), H, None, None)
    qf, kf, vf = qkv.float().view(B, S, 3, H, 32).unbind(2)
    ref = F.scaled_dot_product_attention(qf.transpose(1, 2), kf.transpose(1, 2), vf.transpose(1, 2)).transpose(1, 2)
    assert torch.isfinite(out.float()).all()
    close(out.reshape(B, S, H, 32), ref, what=f"running-max path, growth {growth}")


def test_attention_full_size_properties():
    """Full cfg-2 sequence (S = 4096 tokens, 16 heads, block-causal with 256 electrodes), where the dense oracle is too
    large to run in a test: size-independent properties instead.  (1) block causality is exact: changing keys / values of
    time step >= t leaves the outputs AND the input gradients of all earlier time steps bit-identical, and a loss on the
    earlier time steps sends exactly zero gradient to later tokens; (2) linearity in V; (3) a spot check of 64 random rows against fp32 softmax attention computed row by row."""
    from frankenstein_b200 import ops
    B, S, H, E = 2, 4096, 16, 256
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(11)
    qkv = (torch.randn(B, S, 3 * H * 32, generator=g) * 1.2).to(dev).to(torch.bfloat16)
    mask = ops.LabelMask.block_causal(B, S, E, dev)

    def run(x, w=None):
        xx = x.clone().requires_grad_(True)
        out = ops.attention_qkv(xx * 1.0, H, None, mask)
        if w is None:
            return out.detach(), None
        (out.float() * w).sum().backward()
        return out.detach(), xx.grad.detach()

    w = torch.randn(B, S, H * 32, generator=g).to(dev)
    t0 = 9 * E                                            # boundary between time steps 8 and 9
    w_early = w.clone(); w_early[:, t0:] = 0              # loss that only looks at the earlier time steps
    out_a, grad_a = run(qkv, w_early)
    pert = qkv.clone()
    pert[:, t0:, H * 32:] = (torch.randn(B, S - t0, 2 * H * 32, generator=g) * 1.2).to(dev).to(torch.bfloat16)   # later k and v
    out_b, grad_b = run(pert, w_early)
    assert torch.equal(out_a[:, :t0], out_b[:, :t0]), "outputs of earlier time steps changed with later keys/values"
    assert torch.equal(grad_a[:, :t0], grad_b[:, :t0]), "gradients of earlier tokens changed with later keys/values"
    assert grad_a[:, t0:].abs().max().item() == 0.0, "later tokens received gradient from a loss on earlier time steps"
    # linearity in V
    v2 = qkv.clone(); v2[..., 2 * H * 32:] = (torch.randn(B, S, H * 32, generator=g)).to(dev).to(torch.bfloat16)
    vs = qkv.clone(); vs[..., 2 * H * 32:] = (qkv[..., 2 * H * 32:].float() + v2[..., 2 * H * 32:].float()).to(torch.bfloat16)
    o1, _ = run(qkv); o2, _ = run(v2); o3, _ = run(vs)
    close(o3, o1.float() + o2.float(), rtol=2e-2, what="linearity in V")
    # spot check of random rows against fp32 softmax
    q, k, v = qkv.float().view(B, S, 3, H, 32).unbind(2)
    rows = torch.randint(0, S, (64,), generator=g).tolist()
    for i in rows[:64]:
        b, hh = i % B, i % H
        vis = (torch.arange(S, device=dev) // E) <= (i // E)
        sc = (k[b, :, hh] @ q[b, i, hh]) / math.sqrt(32.0)
        p_ = torch.softmax(sc.masked_fill(~vis, float("-inf")), dim=0)
        ref = p_ @ v[b, :, hh]
        got = o1[b, i].view(H, 32)[hh].float()
        assert (got - ref).abs().max().item() <= 2e-2 * ref.abs().max().item() + 2e-3, f"row {i}"


@pytest.mark.parametrize("per_sample", [False, True])
def test_rope_matches_reference_formula(per_sample):
    from frankenstein_b200 import ops
    from frankenstein_b200.brainformer import build_complex_rope_cache, apply_rope
    B, S, H, P = 2, 100, 3, 256
    g = torch.Generator().manual_seed(1)
    cache = build_complex_rope_cache(32, P, 10000)
    x = torch.randn(B, S, H, 32, generator=g).to(torch.bfloat16)
    if per_sample:
        pos = torch.stack([torch.sort(torch.randperm(P, generator=g)[:S])[0] for _ in range(B)])
        ref = apply_rope(x, cache[pos])
        spec = ops.RopeSpec(torch.view_as_real(cache).float().cuda(), pos.cuda(), 0)
    else:
        ref = apply_rope(x, cache)                      # rope[-S:]
        spec = ops.RopeSpec.from_complex(cache.cuda(), S, last=True)
    xd = x.cuda().clone()
    ops._rope_inplace(xd, spec, False)
    close(xd, ref, rtol=1e-2, what="rope")
    ops._rope_inplace(xd, spec, True)                   # inverse rotation restores the input (bf16 rounding twice)
    close(xd, x, rtol=2e-2, what="rope inverse")


def _small_cfg():
    return dict(window_size=64, n_electrodes=16, patch_size=8, dim=64, n_layers=2, head_dim=32, hidden_dim=128,
                n_heads=2, n_kv_heads=2, n_dec_layers=2, decoder_dim=64)


def _grads_close(model, ref_sd, names, rtol=5e-2):
    for n in names:
        a = dict(model.named_parameters())[n].grad
        b = ref_sd[n].grad
        assert a is not None and b is not None, n
        close(a, b, rtol=rtol, what=f"grad {n}")


def test_encoder_matches_oracle():
    from frankenstein_b200 import brainformer as bf
    from oracle import brainformer_ref as o
    torch.manual_seed(0)
    cfg = _small_cfg()
    enc = bf.Encoder(bf.MAEConfig(**cfg)).cuda()
    x = torch.randn(3, 64, 16)
    w = torch.randn(3, 128, 64)
    y = enc(x.cuda())
    (y * w.cuda()).sum().backward()
    sd = {k: v.detach().cpu().clone().requires_grad_(v.is_floating_point()) for k, v in enc.state_dict().items()}
    yr = o.encoder_forward(sd, x, cfg)
    (yr * w).sum().backward()
    assert y.dtype == torch.float32 and tuple(y.shape) == (3, 128, 64)
    close(y, yr, what="encoder out")
    _grads_close(enc, sd, ["transformer.emb.weight", "space_embedding", "transformer.h.0.attn.qw.weight",
                           "transformer.h.1.mlp.w2.weight", "transformer.h.0.ln_1.weight", "transformer.ln_f.bias"])


def test_mae_matches_oracle():
    from frankenstein_b200 import brainformer as bf
    from oracle import brainformer_ref as o
    torch.manual_seed(1)
    cfg = _small_cfg()
    mae = bf.MAE(bf.MAEConfig(**cfg)).cuda()
    x = torch.randn(2, 64, 16)
    g = torch.Generator().manual_seed(2)
    n_tok = 128
    order = torch.stack([torch.randperm(n_tok, generator=g) for _ in range(2)])
    masked, unmasked = torch.sort(order[:, :96])[0], torch.sort(order[:, 96:])[0]
    mae.get_masking_indices = lambda r, xx: (masked.cuda(), unmasked.cuda())
    loss, _ = mae(x.cuda())
    loss.backward()
    sd = {k: v.detach().cpu().clone().requires_grad_(v.is_floating_point()) for k, v in mae.state_dict().items()}
    lr, _ = o.mae_forward(sd, x, cfg, masked, unmasked)
    lr.backward()
    assert abs(float(loss) - float(lr)) <= RTOL * abs(float(lr)), (float(loss), float(lr))
    _grads_close(mae, sd, ["mask_token", "to_signals.weight", "decoder.h.1.attn.vw.weight", "encoder.transformer.emb.weight",
                           "encoder.transformer.h.0.mlp.w1.weight", "decoder_pos_emb.weight"], rtol=8e-2)


@pytest.mark.skip(reason="CPU known-answer lives in tests/test_cpu.py")
def _unused_param_counts():
    """franky_baseline_gpt2.ipynb:225-229 prints Encoder 4.27M / Full HandFormer 6.32M for window 768, patch 32."""
    from frankenstein_b200 import brainformer as bf
    mc = bf.MAEConfig(window_size=768, patch_size=32)
    enc = bf.Encoder(mc)
    assert round(enc.get_num_params() / 1e6, 2) == 4.27
    assert tuple(enc.attn_mask.shape) == (6144, 6144)
    full = bf.BrainFormer(bf.Config(encoder=mc, n_output_tokens=32, output_dim=768))
    assert round(full.get_num_params() / 1e6, 2) == 6.32
