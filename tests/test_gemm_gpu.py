"""The library's own tcgen05 GEMMs (csrc/gemm.cu) against plain PyTorch fp32 matmuls of the same bf16 operands: the NT
kernels (A-resident for K <= 512, streaming for longer K), their fused epilogues (bias, RoPE, SwiGLU gate) and the TN weight-gradient kernel (MN-major operands, split reduction), then the autograd Functions built on them."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def close(a, b, rtol, what=""):
    a, b = a.float().cpu(), b.float().cpu()
    scale = b.abs().max().item() + 1e-12
    err = (a - b).abs().max().item()
    assert err <= rtol * scale, f"{what}: max err {err:.4g} vs scale {scale:.4g}"


def _rand(shape, g, scale=1.0):
    return (torch.randn(*shape, generator=g) * scale).cuda().to(torch.bfloat16)


@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (1000, 512, 512), (300, 1536, 512), (4173, 96, 200), (517, 512, 32),
                                   (40000, 512, 512), (64, 32, 8),                       # A-resident kernel
                                   (1000, 512, 2048), (513, 512, 4096), (300, 96, 1536), (2048, 768, 520)])   # streaming kernel
@pytest.mark.parametrize("with_bias", [False, True])
def test_gemm_nt_matches_fp32_matmul(M, N, K, with_bias):
    from frankenstein_b200 import gemm
    g = torch.Generator().manual_seed(M + N + K)
    a, b = _rand((M, K), g), _rand((N, K), g, 0.5)
    bias = torch.randn(N, generator=g).cuda() if with_bias else None
    c = gemm.gemm_nt(a, b, bias)
    ref = a.float() @ b.float().t()
    if with_bias:
        ref = ref + bias
    assert c.shape == (M, N) and c.dtype == torch.bfloat16
    close(c, ref, 1e-2, f"gemm_nt {M}x{N}x{K}")


def test_gemm_nt_strided_operand():
    """A with a leading dimension larger than K (a column slice of a wider activation buffer)."""
    from frankenstein_b200 import gemm
    g = torch.Generator().manual_seed(3)
    wide = _rand((700, 1536), g)
    a = wide[:, 512:1024]
    b = _rand((256, 512), g)
    close(gemm.gemm_nt(a, b), a.float() @ b.float().t(), 1e-2, "strided A")


@pytest.mark.parametrize("per_sample", [False, True])
def test_gemm_rope_epilogue(per_sample):
    """q | k columns rotated as apply_rope (models/brainformer.py:70-91) does, v columns untouched."""
    from frankenstein_b200 import gemm
    from frankenstein_b200.brainformer import build_complex_rope_cache
    from frankenstein_b200.ops import RopeSpec
    g = torch.Generator().manual_seed(9)
    B, S, D, H = 3, 200, 128, 4
    inner = H * 32
    x, w = _rand((B * S, D), g), _rand((3 * inner, D), g, 0.3)
    cache = build_complex_rope_cache(32, 512, 10000.0).cuda()
    table = torch.view_as_real(cache).float().contiguous()
    if per_sample:
        pos = torch.stack([torch.sort(torch.randperm(512, generator=g)[:S])[0] for _ in range(B)]).cuda()
        spec = RopeSpec(table, pos, 0)
    else:
        pos = (torch.arange(S) + (512 - S))[None].expand(B, S).cuda()
        spec = RopeSpec(table, None, 512 - S)
    out = gemm.gemm_nt(x, w, None, gemm.EPI_ROPE, rope=spec, rope_cols=2 * inner, rope_S=S)
    ref = (x.float() @ w.float().t()).view(B, S, 3, H, 16, 2)
    rot = torch.view_as_real(torch.view_as_complex(ref[:, :, :2].contiguous()) * cache[pos][:, :, None, None, :])
    ref = torch.cat([rot, ref[:, :, 2:]], dim=2).reshape(B * S, 3 * inner)
    close(out, ref, 1e-2, "rope epilogue")


@pytest.mark.parametrize("M,D,H", [(300, 64, 128), (1000, 512, 2048), (129, 256, 384)])
def test_gemm_swiglu_gate_epilogue(M, D, H):
    """The w1 | w3 projection with the gate in its epilogue: h13 interleaved in blocks of 128 and gated = silu(h1) * h3."""
    from frankenstein_b200 import gemm
    g = torch.Generator().manual_seed(M)
    x = _rand((M, D), g)
    w1, w3 = _rand((H, D), g, D ** -0.5), _rand((H, D), g, D ** -0.5)
    w13 = gemm._interleave(w1, w3)
    h13, gated = gemm.gemm_nt(x, w13, None, gemm.EPI_SWIGLU)
    h1_ref, h3_ref = x.float() @ w1.float().t(), x.float() @ w3.float().t()
    a, b = gemm._deinterleave(h13.t().contiguous())          # de-interleave along the column axis
    close(a.t(), h1_ref, 1e-2, "h1")
    close(b.t(), h3_ref, 1e-2, "h3")
    close(gated, F.silu(h1_ref) * h3_ref, 2e-2, "gated")


@pytest.mark.parametrize("M", [300, 4173])          # 3 row blocks: single-CTA kernel; 33 row blocks: CTA pairs
@pytest.mark.parametrize("epi", ["store", "store_bias", "rope32", "rope64", "swiglu"])
def test_a_resident_epilogues(epi, M):
    """Every epilogue on both A-resident kernels (K <= 512), with a partial last row block and, but for SwiGLU, a partial
    last column tile; RoPE positions are (m % S) + offset."""
    from frankenstein_b200 import gemm
    from frankenstein_b200.brainformer import build_complex_rope_cache
    from frankenstein_b200.ops import RopeSpec
    g = torch.Generator().manual_seed(M)
    K, inner, S, off = 256, 128, M // 3, 7
    x = _rand((M, K), g)
    if epi == "swiglu":
        w1, w3 = _rand((256, K), g, K ** -0.5), _rand((256, K), g, K ** -0.5)
        h13, gated = gemm.gemm_nt(x, gemm._interleave(w1, w3), None, gemm.EPI_SWIGLU)
        h1, h3 = x.float() @ w1.float().t(), x.float() @ w3.float().t()
        close(h13, gemm._interleave(h1.t(), h3.t()).t(), 1e-2, "h13")
        close(gated, F.silu(h1) * h3, 2e-2, "gated")
        return
    w = _rand((3 * inner, K), g, K ** -0.5)
    ref = x.float() @ w.float().t()
    if epi.startswith("store"):
        bias = torch.randn(3 * inner, generator=g).cuda() if epi == "store_bias" else None
        out = gemm.gemm_nt(x, w, bias)
        if bias is not None:
            ref = ref + bias
    else:
        hd = 32 if epi == "rope32" else 64
        cache = build_complex_rope_cache(hd, 2048, 10000.0).cuda()
        out = gemm.gemm_nt(x, w, None, gemm.ROPE_EPILOGUE[hd], rope=RopeSpec(torch.view_as_real(cache).float(), None, off),
                           rope_cols=2 * inner, rope_S=S)
        pos = torch.arange(M, device="cuda") % S + off
        qk = torch.view_as_complex(ref[:, :2 * inner].reshape(M, 2 * inner // hd, hd // 2, 2).contiguous())
        ref[:, :2 * inner] = torch.view_as_real(qk * cache[pos][:, None, :]).reshape(M, 2 * inner)
    assert out.shape == (M, 3 * inner)
    close(out, ref, 1e-2, f"{epi} M={M}")


def test_removed_swiglu_backward_epilogue_is_rejected():
    """Epilogue 3 (the SwiGLU backward, removed) fails on the host, before anything is launched."""
    from frankenstein_b200._lib import FkError, check, launch_count, lib, ptr, stream
    a, b = torch.zeros(256, 64, device="cuda", dtype=torch.bfloat16), torch.zeros(256, 64, device="cuda", dtype=torch.bfloat16)
    c, c2 = torch.empty(256, 256, device="cuda", dtype=torch.bfloat16), torch.empty(256, 512, device="cuda", dtype=torch.bfloat16)
    n0 = launch_count()
    with pytest.raises(FkError, match="removed"):
        check(lib().fk_gemm_nt(ptr(a), 64, ptr(b), 64, ptr(c), 256, 256, 256, 64, None, 3, ptr(c2), 512, None, 0, None, 0,
                               0, 0, stream()), "fk_gemm_nt")
    assert launch_count() == n0


@pytest.mark.parametrize("M,Na,Nb", [(1000, 512, 512), (4096, 1536, 512), (333, 64, 64), (70000, 4096, 512), (64, 128, 192),
                                     (5000, 512, 2048), (100, 320, 448)])
def test_gemm_tn_matches_fp32_matmul(M, Na, Nb):
    from frankenstein_b200 import gemm
    g = torch.Generator().manual_seed(M + Na)
    a, b = _rand((M, Na), g), _rand((M, Nb), g)
    out = gemm.gemm_tn(a, b)
    ref = a.float().t() @ b.float()
    assert out.dtype == torch.float32 and out.shape == (Na, Nb)
    close(out, ref, 2e-3, f"gemm_tn {M}x{Na}x{Nb}")
    assert torch.equal(out, gemm.gemm_tn(a, b)), "the split reduction must be bit-reproducible"


@pytest.mark.parametrize("head_dim", [32, 64])
def test_linear_qkv_mlp_functions(head_dim):
    """The autograd Functions (forward + all gradients) against fp32 PyTorch on the same weights: linear, the SwiGLU MLP
    (backward: d-gated GEMM, then the streaming SwiGLU derivative) and the fused q | k | v projection with the RoPE
    epilogue of the given head width."""
    from frankenstein_b200 import gemm
    from frankenstein_b200.brainformer import apply_rope, build_complex_rope_cache
    from frankenstein_b200.ops import RopeSpec
    g = torch.Generator().manual_seed(0)
    B, S, D, H, NH = 2, 300, 128, 256, 4
    inner = NH * head_dim
    x = torch.randn(B, S, D, generator=g).cuda()
    wout = torch.randn(B, S, D, generator=g).cuda()

    def params(*shape, s):
        return (torch.randn(*shape, generator=g) * s).cuda().requires_grad_(True)

    # ---- linear ----
    w, bias = params(D, D, s=D ** -0.5), params(D, s=0.1)
    xr = x.clone().requires_grad_(True)
    (gemm.linear(xr, w, bias).float() * wout).sum().backward()
    w2, b2, x2 = w.detach().clone().requires_grad_(True), bias.detach().clone().requires_grad_(True), x.clone().requires_grad_(True)
    (F.linear(x2, w2, b2) * wout).sum().backward()
    close(xr.grad, x2.grad, 2e-2, "linear dx"); close(w.grad, w2.grad, 2e-2, "linear dw"); close(bias.grad, b2.grad, 2e-2, "linear db")
    # ---- swiglu mlp ----
    w1, w3, wd = params(H, D, s=D ** -0.5), params(H, D, s=D ** -0.5), params(D, H, s=H ** -0.5)
    xr = x.clone().requires_grad_(True)
    y = gemm.swiglu_mlp(xr, w1, w3, wd)
    (y.float() * wout).sum().backward()
    ref_p = [t.detach().clone().requires_grad_(True) for t in (x, w1, w3, wd)]
    yr = F.linear(F.silu(F.linear(ref_p[0], ref_p[1])) * F.linear(ref_p[0], ref_p[2]), ref_p[3])
    (yr * wout).sum().backward()
    close(y, yr, 2e-2, "mlp out")
    for name, a, b in (("dx", xr, ref_p[0]), ("dw1", w1, ref_p[1]), ("dw3", w3, ref_p[2]), ("dw2", wd, ref_p[3])):
        close(a.grad, b.grad, 3e-2, f"mlp {name}")
    # ---- qkv + rope ----
    wq, wk, wv = (params(inner, D, s=D ** -0.5) for _ in range(3))
    cache = build_complex_rope_cache(head_dim, 512, 10000.0).cuda()
    spec = RopeSpec.from_complex(cache, S, last=True)
    wq_out = torch.randn(B, S, 3 * inner, generator=g).cuda()
    xr = x.clone().requires_grad_(True)
    qkv = gemm.qkv_rope(xr, wq, wk, wv, spec, NH)
    ref_p = [t.detach().clone().requires_grad_(True) for t in (x, wq, wk, wv)]
    q = apply_rope(F.linear(ref_p[0], ref_p[1]).view(B, S, NH, head_dim), cache).reshape(B, S, inner)
    k = apply_rope(F.linear(ref_p[0], ref_p[2]).view(B, S, NH, head_dim), cache).reshape(B, S, inner)
    ref = torch.cat([q, k, F.linear(ref_p[0], ref_p[3])], dim=-1)
    close(qkv, ref, 2e-2, "qkv rope out")
    # the Function's backward takes the gradient w.r.t. the UNROTATED projection (the attention backward un-rotates dq / dk):
    qkv.backward(wq_out.to(torch.bfloat16))
    plain = torch.cat([F.linear(ref_p[0], ref_p[i]) for i in (1, 2, 3)], dim=-1)
    (plain * wq_out.to(torch.bfloat16).float()).sum().backward()
    close(xr.grad, ref_p[0].grad, 2e-2, "qkv dx")
    for name, a, b in (("dwq", wq, ref_p[1]), ("dwk", wk, ref_p[2]), ("dwv", wv, ref_p[3])):
        close(a.grad, b.grad, 2e-2, f"qkv {name}")


@pytest.mark.parametrize("B,T,E,patch,dim", [(2, 64, 64, 32, 128), (3, 96, 128, 48, 64), (2, 512, 256, 32, 512), (1, 64, 192, 16, 320),
                                             (2, 128, 64, 64, 64)])
def test_patch_embed_matches_linear_of_to_patches(B, T, E, patch, dim):
    """fk_patch_embed_forward (TMA-strided patchify + tcgen05 contraction + bias) against F.linear(to_patches(x)) in fp32 on
    the same bf16-rounded operands (models/brainformer.py:282-285), with dW / db through the split-K TN kernel."""
    from frankenstein_b200 import gemm
    g = torch.Generator().manual_seed(T + E)
    x = torch.randn(B, T, E, generator=g).cuda()
    w = (torch.randn(dim, patch, generator=g) * patch ** -0.5).cuda().requires_grad_(True)
    b = (torch.randn(dim, generator=g) * 0.1).cuda().requires_grad_(True)
    wout = torch.randn(B, (T // patch) * E, dim, generator=g).cuda().to(torch.bfloat16)
    y = gemm.patch_embed(x, w, b)
    y.backward(wout)
    xr = x.to(torch.bfloat16).float()
    patches = xr.view(B, T // patch, patch, E).transpose(2, 3).reshape(B, (T // patch) * E, patch)
    w2, b2 = w.detach().to(torch.bfloat16).float().requires_grad_(True), b.detach().clone().requires_grad_(True)
    ref = F.linear(patches, w2, b2)
    (ref * wout.float()).sum().backward()
    assert y.shape == ref.shape and y.dtype == torch.bfloat16
    close(y, ref, 1e-2, "patch embed out")
    close(w.grad, w2.grad, 2e-2, "patch embed dw")
    close(b.grad, b2.grad, 2e-2, "patch embed db")
