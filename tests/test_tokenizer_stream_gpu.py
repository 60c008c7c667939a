"""Streaming SoundStream tokenizer (SoundStream.stream): the row-assembly kernel fk_conv_stream_rows against torch bit for
bit, the GEMM and the codebook search at the handful of rows a batch-1 step gives them, and TokenizerStream against the
offline eval path (get_quantize_vectors, Decoder.forward) and the fp32 oracle over long streams.

Token checks: at least 99.9 % of the indices agree, every disagreement is a near-tie (relative distance gap below 1e-3
under the features of the path compared with), and `quantized` is bit-equal on the rows that agree.  Against the oracle's
fully fp32 encoder the bound is looser (see test_tokens_match_oracle).  Each comparison prints its worst figures
(`pytest -s`).  Inputs are smoothed noise without zero-padded tails: a codebook k-means-initialised on padding holds many
identical codewords, and which of those exact duplicates the search returns depends on its row count, offline as well.
"""
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import index_agreement

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
BINS = 4096
UNEVEN = [8, 4, 20, 4, 60, 12, 128, 44, 4, 16]


def _counters_zero():
    from frankenstein_b200 import _lib
    torch.cuda.synchronize()
    return all(int(t.abs().sum()) == 0 for t in _lib._counter_sets.values())


def _steps(kind, total=BINS):
    if kind == "4":
        return [4] * (total // 4)
    if kind == "32":
        return [32] * (total // 32)
    out, i = [], 0
    while sum(out) < total:
        out.append(min(UNEVEN[i % len(UNEVEN)], total - sum(out)))
        i += 1
    return out


# ------------------------------------------------------------------------------------------------
# kernel
# ------------------------------------------------------------------------------------------------
def _rows_ref(x, r, elu, hist, rpt, total):
    """torch: [hist | act(x + r)] per trial at rows [0, h + n) of rpt, zeros elsewhere; and the last h rows"""
    B, n, C = x.shape
    if r is not None:
        s = (x.float() + r.float()).to(BF16)
    else:
        s = x
    if elu:
        s = F.elu(s)
    new = s.to(BF16)
    full = new if hist is None else torch.cat([hist, new], 1)
    buf = torch.zeros(total, C, device=x.device, dtype=BF16)
    buf[:B * rpt].view(B, rpt, C)[:, :full.shape[1]] = full
    return buf, (None if hist is None else full[:, full.shape[1] - hist.shape[1]:])


def _launch_rows(x, r, elu, hist_in, hist_out, rpt, total, C):
    from frankenstein_b200 import conv
    from frankenstein_b200._lib import lib, ptr, stream
    B, n, _ = x.shape
    h = 0 if hist_in is None else hist_in.shape[1]
    out = torch.full((total, C), 7.0, device=x.device, dtype=BF16)              # every row must be written
    rs = (0, 0) if r is None else conv._row_strides(r)
    rc = lib().fk_conv_stream_rows(ptr(x), 0 if x.dtype == torch.float32 else 1, *conv._row_strides(x), ptr(r), *rs,
                                   ptr(hist_in), ptr(hist_out), B, n, h, C, int(elu), ptr(out), rpt, total, stream())
    return rc, out


@pytest.mark.parametrize("dtype", [torch.float32, BF16])
@pytest.mark.parametrize("res", [False, True])
@pytest.mark.parametrize("elu", [False, True])
@pytest.mark.parametrize("h", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("B,n,C,strided", [(3, 1, 64, False), (2, 2, 256, True), (1, 5, 8, False), (4, 37, 128, True)])
def test_stream_rows_bit_exact(dtype, res, elu, h, B, n, C, strided):
    g = torch.Generator().manual_seed(B * 100 + n * 10 + h)
    pad = 24 if strided else 0                                      # row-strided views, as the sliced GEMM outputs are
    x = (torch.randn(B, n + 3, C + pad, generator=g) * 3).cuda().to(dtype)[:, 1:n + 1, :C]
    r = (torch.randn(B, n + 2, C + pad, generator=g) * 2).cuda().to(BF16)[:, 2:, :C] if res else None
    if r is not None:
        r[0, 0, :8] = torch.tensor([0.0, -0.0, 1e-30, -1e-30, -80.0, 80.0, -1e-3, 3.0], dtype=BF16)
    x[0, 0, :8] = torch.tensor([0.0, -0.0, 1e-30, -1e-30, -88.0, 1e4, -1e-3, -0.5], dtype=dtype)
    hist_in = (torch.randn(B, h, C, generator=g)).cuda().to(BF16) if h else None
    hist_out = torch.full((B, h, C), 5.0, device="cuda", dtype=BF16) if h else None
    s = 2 if h == 3 else 1
    rpt = -(-(n + h) // s) * s + (1 if n == 2 else 0)
    total = B * rpt + h + 1
    rc, out = _launch_rows(x, r, elu, hist_in, hist_out, rpt, total, C)
    assert rc == 0
    ref, ref_hist = _rows_ref(x, r, elu, hist_in, rpt, total)
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))
    if h:
        assert torch.equal(hist_out.view(torch.int16), ref_hist.view(torch.int16))


def test_stream_rows_rejections():
    from frankenstein_b200 import conv
    from frankenstein_b200._lib import lib, ptr, stream
    x = torch.randn(2, 4, 64, device="cuda", dtype=BF16)
    hi, ho = torch.zeros(2, 2, 64, device="cuda", dtype=BF16), torch.zeros(2, 2, 64, device="cuda", dtype=BF16)
    out = torch.empty(40, 64, device="cuda", dtype=BF16)

    def call(x_dtype=1, n=4, h=2, C=64, act=1, hin=hi, hout=ho, rpt=6, total=12, st=64):
        return lib().fk_conv_stream_rows(ptr(x), x_dtype, 256, st, None, 0, 0, ptr(hin), ptr(hout), 2, n, h, C, act,
                                         ptr(out), rpt, total, stream())
    assert call() == 0
    for bad in (dict(x_dtype=2), dict(n=0), dict(C=60), dict(act=2), dict(hin=None), dict(hout=hi), dict(rpt=5),
                dict(total=11), dict(st=60)):
        assert call(**bad) != 0, bad
    with pytest.raises(conv.FkError):
        conv._row_strides(x.transpose(1, 2))


# ------------------------------------------------------------------------------------------------
# the GEMM and the search at the row counts of a batch-1 step
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("K", [192, 2560])
def test_gemm_nt_few_rows(M, K):
    """implicit-GEMM operand with M overlapping rows (row stride 64 elements, K up to the streaming kernel's range)"""
    from frankenstein_b200 import gemm
    g = torch.Generator().manual_seed(M * K)
    step = 64
    buf = torch.randn(M * step + K, 1, generator=g).view(-1).cuda().to(BF16)
    A = torch.as_strided(buf, (M, K), (step, 1))
    W = (torch.randn(256, K, generator=g) * K ** -0.5).cuda().to(BF16)
    bias = torch.randn(256, generator=g).cuda()
    y = gemm.gemm_nt(A, W, bias)
    ref = A.double() @ W.double().t() + bias.double()
    assert y.shape == (M, 256)
    assert (y.double() - ref).abs().max().item() <= 1e-2 * ref.abs().max().item()


@pytest.mark.parametrize("N", [1, 2, 3, 8])
@pytest.mark.parametrize("K,cosine", [(512, True), (8192, False)])
def test_search_few_rows(N, K, cosine):
    """search + finish with 1 to 8 rows return the exact nearest codeword of the fp32 rows"""
    from frankenstein_b200 import vector_quantize as vq
    g = torch.Generator().manual_seed(N + K)
    D = 256 if K == 8192 else 64
    e = torch.randn(N, D, generator=g)
    C = torch.randn(K, D, generator=g)
    if cosine:
        C = F.normalize(C, dim=-1)
    xn, xb, _ = vq.prepare_input(e.cuda(), cosine)
    cb, c2 = vq.prepare_codebook(C.cuda(), cosine)
    cv, ci = vq.search(xb, cb, c2, K, cosine)
    ind, q, _ = vq.finish(xn, C.cuda(), cv, ci, cosine, False, 0.0)
    x = xn.cpu().double()
    score = x @ C.double().t() if cosine else -torch.cdist(x, C.double())
    ref = score.argmax(1)
    agree, worst = index_agreement(ind, ref, x.float(), C, cosine)
    assert agree == 1.0 or worst < 1e-3, (agree, worst)
    assert torch.equal(q.cpu(), C[ind.cpu()])
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# TokenizerStream
# ------------------------------------------------------------------------------------------------
_MODELS = {}


def _signal(B, T, C, seed):
    """smoothed, per-channel z-scored noise [B, T, C] (tests.helpers.synth_trials without its zero-padded tails)"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T + 4, C, generator=g)
    x = sum(x[:, i:T + i] for i in range(5)) / 5.0
    return ((x - x.mean(dim=1, keepdim=True)) / x.std(dim=1, keepdim=True)).contiguous()


def _model(C, cosine):
    """an eval SoundStream whose codebook was k-means initialised on its own features (one training forward)"""
    key = (C, cosine)
    if key not in _MODELS:
        from frankenstein_b200.vq_brain import SoundStream
        torch.manual_seed(C + cosine)
        E = 64 if C == 64 else 128
        m = SoundStream(C=C, D=64, codebook_size=512, n_electrodes=E, use_cosine_sim=cosine).cuda()
        m.train()
        with torch.no_grad():
            m(_signal(8, T=512, C=E, seed=7).cuda())
        m.eval()
        _MODELS[key] = m
    return _MODELS[key]


def _stream_all(m, x, steps, reconstruct=False):
    s = m.stream(x.shape[0], reconstruct=reconstruct)
    outs, t = [], 0
    for n in steps:
        outs.append(s.step(x[:, t:t + n]))
        t += n
    assert s.length == t
    return s, [torch.cat([o[i] for o in outs], 1) for i in range(len(outs[0]))]


def _check_tokens(ind, q, ref_ind, ref_q, feats, embed, cosine, what):
    agree, worst = index_agreement(ind, ref_ind, feats.reshape(-1, feats.shape[-1]).float().cpu(), embed.cpu(), cosine)
    same = (ind == ref_ind)
    print(f"{what}: index agreement {agree:.6f}, worst near-tie gap {worst:.3g}, "
          f"quantized max |diff| on agreeing rows {(q[same] - ref_q[same]).abs().max().item() if same.any() else 0.0:.3g}")
    assert agree >= 0.999, f"{what}: index agreement {agree}"
    assert worst < 1e-3, f"{what}: a mismatch is not a near-tie (gap {worst})"
    assert torch.equal(q[same], ref_q[same]), f"{what}: quantized differs on agreeing rows"


@pytest.mark.parametrize("C", [64, 256])
@pytest.mark.parametrize("cosine", [False, True])
@pytest.mark.parametrize("B", [1, 3, 32])
def test_tokens_match_offline_eval(C, cosine, B):
    m = _model(C, cosine)
    x = _signal(B, T=BINS, C=m.encoder.layers[0].in_channels, seed=B + C).cuda()
    with torch.no_grad():
        ref_ind, ref_q = m.get_quantize_vectors(x)
        feats = m.encoder(x)
    embed = m.quantizer.codebook
    kinds = ("4", "32", "uneven") if B != 3 else ("32", "uneven")
    for kind in kinds:
        _, (ind, q) = _stream_all(m, x, _steps(kind))
        assert ind.shape == (B, BINS // 4) and ind.dtype == torch.int64 and q.dtype == torch.float32
        _check_tokens(ind, q, ref_ind, ref_q, feats, embed, cosine, f"C {C} cos {cosine} B {B} steps {kind} vs offline")
    assert _counters_zero()


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return ((a - b).norm() / b.norm()).item()


@pytest.mark.parametrize("C", [64, 256])
@pytest.mark.parametrize("cosine", [False, True])
def test_tokens_match_oracle(C, cosine):
    """The stream's encoder features (bit-equal to Encoder.forward, within 2e-2 of the oracle's encoder_forward) and its
    tokens against the fp32 oracle quantizer: the full token checks on the stream's features; on the oracle's own fp32
    features the activations' bf16 rounding moves tokens that are within about 1e-2 of a tie (measured: 98.8 - 99.3 %
    agreement, worst gap 3.6e-3), for the offline path exactly as for the stream."""
    from oracle.soundstream_ref import encoder_forward
    from oracle.vector_quantize_ref import VectorQuantizeRef
    m = _model(C, cosine)
    B = 3
    x = _signal(B, T=BINS, C=m.encoder.layers[0].in_channels, seed=11 + C).cuda()
    s, (ind, q) = _stream_all(m, x, _steps("uneven"))
    s.reset()                                                # the same steps again, keeping the encoder's features
    feats, t = [], 0
    with torch.no_grad():
        for n in _steps("uneven"):
            feats.append(s._run(s._layers[0], x[:, t:t + n]))
            s._cur ^= 1
            t += n
        feats = torch.cat(feats, 1)
        assert torch.equal(feats, m.encoder(x))
    sd = {k: v.detach().float().cpu() for k, v in m.state_dict().items()}
    vq = VectorQuantizeRef(dim=64, codebook_size=512, commitment_weight=0.25, use_cosine_sim=cosine).eval()
    vq._codebook.embed.copy_(m.quantizer.codebook.cpu()[None])
    with torch.no_grad():
        e_ref = encoder_forward(sd, x.cpu())
        err = _rel(feats, e_ref)
        q_ref, i_ref, _ = vq(feats.float().cpu())
        q_fp32, i_fp32, _ = vq(e_ref)
    print(f"C {C} cos {cosine}: stream features vs encoder_forward relative error {err:.3g}")
    assert err <= 2e-2
    _check_tokens(ind.cpu(), q.cpu(), i_ref, q_ref.float(), feats, m.quantizer.codebook, cosine,
                  f"C {C} cos {cosine} vs oracle quantizer")
    agree, worst = index_agreement(ind.cpu(), i_fp32, e_ref.reshape(-1, 64), m.quantizer.codebook.cpu(), cosine)
    same = ind.cpu() == i_fp32
    print(f"C {C} cos {cosine} vs oracle encoder + quantizer (fp32 features): index agreement {agree:.6f}, "
          f"worst gap {worst:.3g}")
    assert agree >= 0.98 and worst < 1e-2 and torch.equal(q.cpu()[same], q_fp32[same])
    assert _counters_zero()


@pytest.mark.parametrize("C", [64, 256])
def test_decoder_reconstruction(C):
    from oracle.soundstream_ref import decoder_forward
    m = _model(C, False)
    x = _signal(3, T=1024, C=m.encoder.layers[0].in_channels, seed=5).cuda()
    _, (ind, q, o) = _stream_all(m, x, _steps("uneven", 1024), reconstruct=True)
    assert o.shape == x.shape
    with torch.no_grad():
        off = m.decoder(q)                                   # the stream's own codes: index flips cannot hide an error
    sd = {k: v.detach().float().cpu() for k, v in m.state_dict().items()}
    ref = decoder_forward(sd, q.cpu())
    e_off, e_ref = _rel(o, off), _rel(o, ref)
    print(f"decoder C {C}: relative error vs Decoder.forward {e_off:.3g}, vs oracle {e_ref:.3g}")
    assert e_off <= 1e-2 and e_ref <= 2e-2
    assert _counters_zero()


def test_state_errors_reset_and_snapshot():
    from frankenstein_b200._lib import FkError
    m = _model(64, True)
    x = _signal(2, T=256, C=64, seed=3).cuda()
    steps = [8, 4, 20, 4, 60, 32, 128]

    def run(s, rejects=False):
        outs, t = [], 0
        for i, n in enumerate(steps):
            if rejects and i in (1, 4):
                L = s.length
                for bad in (x[:, t:t + 6],                          # not a multiple of 4
                            x[:, t:t],                              # no bins
                            x[:1, t:t + 4],                         # batch size
                            x[:, t:t + 4, :32],                     # channel count
                            x[:, t:t + 4].cpu(),                    # CPU tensor
                            x[:, t:t + 4].half(),                   # dtype
                            x[0]):                                  # rank
                    with pytest.raises(FkError):
                        s.step(bad)
                    assert s.length == L
            outs.append(s.step(x[:, t:t + n]))
            t += n
        return [torch.cat([o[i] for o in outs], 1) for i in range(3)]

    s = m.stream(2, reconstruct=True)
    ref = run(s)
    clean = run(m.stream(2, reconstruct=True))
    assert all(torch.equal(a, b) for a, b in zip(ref, clean))
    # rejected steps leave the state unchanged
    got = run(m.stream(2, reconstruct=True), rejects=True)
    assert all(torch.equal(a, b) for a, b in zip(ref, got))
    # reset == a fresh stream
    s.reset()
    assert s.length == 0
    assert all(torch.equal(a, b) for a, b in zip(ref, run(s)))
    # the stream is a snapshot: changing the model afterwards does not change it
    s2 = m.stream(2, reconstruct=True)
    saved = {k: v.clone() for k, v in m.state_dict().items()}
    try:
        with torch.no_grad():
            for p in m.parameters():
                p.add_(0.5)
            m.quantizer._codebook.embed.mul_(-1.0)
            m.quantizer._mark_dirty()
        assert all(torch.equal(a, b) for a, b in zip(ref, run(s2)))
    finally:
        m.load_state_dict(saved)
    assert _counters_zero()


def test_stream_ignores_training_mode():
    m = _model(64, False)
    x = _signal(2, T=128, C=64, seed=9).cuda()
    _, ref = _stream_all(m, x, [16] * 8)
    cb = m.quantizer._codebook
    before = [t.clone() for t in (cb.embed, cb.embed_avg, cb.cluster_size)]
    m.train()
    try:
        _, got = _stream_all(m, x, [16] * 8)
    finally:
        m.eval()
    assert all(torch.equal(a, b) for a, b in zip(ref, got))
    assert all(torch.equal(a, b) for a, b in zip(before, (cb.embed, cb.embed_avg, cb.cluster_size)))


def test_two_streams_on_two_cuda_streams():
    m = _model(256, False)
    xs = [_signal(3, T=512, C=128, seed=s).cuda() for s in (1, 2)]
    steps = _steps("uneven", 512)
    serial = [_stream_all(m, x, steps, reconstruct=True)[1] for x in xs]
    streams = [m.stream(3, reconstruct=True) for _ in xs]
    cs = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()
    outs, t = [[], []], 0
    for n in steps:
        for i in (0, 1):
            with torch.cuda.stream(cs[i]):
                outs[i].append(streams[i].step(xs[i][:, t:t + n]))
        t += n
    torch.cuda.synchronize()
    for i in (0, 1):
        got = [torch.cat([o[j] for o in outs[i]], 1) for j in range(3)]
        assert all(torch.equal(a, b) for a, b in zip(got, serial[i]))
    assert _counters_zero()


def test_rejections_at_creation():
    from frankenstein_b200._lib import FkError
    from frankenstein_b200.vq_brain import SoundStream
    fresh = SoundStream(C=64, D=64, codebook_size=128, n_electrodes=64).cuda().eval()
    with pytest.raises(FkError, match="not initialised"):
        fresh.stream(1)
    narrow = SoundStream(C=48, D=64, codebook_size=128, n_electrodes=64).cuda().eval()
    narrow.quantizer._codebook.initted.fill_(1.0)
    narrow.quantizer._mark_dirty()
    with pytest.raises(FkError, match="cuDNN"):
        narrow.stream(1)
    with pytest.raises(FkError):
        _model(64, False).stream(0)


def test_no_fallback(monkeypatch):
    from frankenstein_b200 import conv
    m = _model(64, True)
    x = _signal(2, T=64, C=64, seed=4).cuda()
    s = m.stream(2, reconstruct=True)

    def refuse(*a, **k):
        raise AssertionError("cuDNN / torch convolution, _padded or torch ELU used on the stream path")
    for name in ("conv1d", "conv2d", "conv_transpose1d", "conv_transpose2d", "elu"):
        monkeypatch.setattr(F, name, refuse)
    monkeypatch.setattr(conv, "_padded", refuse)
    for t in range(0, 64, 16):
        ind, q, o = s.step(x[:, t:t + 16])
        assert ind.shape == (2, 4) and o.shape == (2, 16, 64)
