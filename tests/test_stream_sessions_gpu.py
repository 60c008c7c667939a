"""Streams whose batch rows are independent sessions: the per-row key counts of the perceiver's cached attention
(fk_small_attn_forward with k_len) against a float64 reference, the per-step positions kernel (fk_stream_positions)
against torch, and Encoder / BrainFormer / SoundStream streams with rows that start, reset and run at different positions,
each row against the offline forward on its own bins, and bit for bit against the same row in a stream whose other rows
do something else.
"""
import pytest
import torch

from tests.test_encoder_stream_gpu import CFG2, _counters_zero, _enc_cfg, _no_dense_attention, rel_close

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16


# ------------------------------------------------------------------------------------------------
# kernel: per-row key counts of the perceiver's cached attention
# ------------------------------------------------------------------------------------------------
def _kv_operands(B, Tq, S, H, hd, seed):
    g = torch.Generator().manual_seed(seed)
    q = (torch.randn(B, Tq, H * hd, generator=g) * 1.5).to(BF16).cuda()
    kv = torch.randn(B, S, 2 * H * hd, generator=g)
    kv[..., :H * hd] *= 1.5
    return q, kv.to(BF16).cuda()


def _kv_reference(q, kv, H, k_len):
    """float64 softmax(q k^T / sqrt(hd)) v of each row over its first k_len[b] keys -> [B, Tq, H, hd] (zeros for 0 keys)"""
    B, Tq, W = q.shape
    hd = W // H
    out = torch.zeros(B, Tq, H, hd, dtype=torch.float64)
    for b in range(B):
        n = int(k_len[b])
        if n == 0:
            continue
        qd = q[b].double().cpu().view(Tq, H, hd)
        kd = kv[b, :n, :W].double().cpu().view(n, H, hd)
        vd = kv[b, :n, W:].double().cpu().view(n, H, hd)
        p = torch.softmax(torch.einsum("qhd,khd->hqk", qd, kd) * hd ** -0.5, dim=-1)
        out[b] = torch.einsum("hqk,khd->qhd", p, vd)
    return out


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_small_attention_k_len_matches_fp64(hd):
    from frankenstein_b200 import ops
    H, Tq, S = 2, 8, 1000                                   # 4 chunks of 256 keys, the last one partial
    counts = [1, 255, 256, 257, 600, S, 0]
    B = len(counts)
    q, kv = _kv_operands(B, Tq, S, H, hd, seed=hd)
    k_len = torch.tensor(counts, dtype=torch.int32).cuda()
    with torch.no_grad():
        out = ops.small_attention_kv_cached(q, kv, H, k_len=k_len)
    ref = _kv_reference(q, kv, H, counts)
    o = out.view(B, Tq, H, hd).double().cpu()
    vmax = kv[..., H * hd:].double().abs().amax().item()
    for b, n in enumerate(counts):
        if n == 0:
            assert bool((o[b] == 0).all()), "a row with no key is not a zero row"
        else:
            err = (o[b] - ref[b]).abs().max().item()
            assert err <= 1e-2 * vmax, f"hd {hd} k_len {n}: max error {err:.3g}"
    assert _counters_zero()


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_small_attention_k_len_bits(hd):
    """row b's bits depend only on its first k_len[b] keys: not on the keys past it, not on other rows' counts, not on
    how many empty chunks follow; k_len = S everywhere is k_len = None"""
    from frankenstein_b200 import ops
    H, Tq, S = 4, 32, 1000
    counts = [300, 1000, 0, 513, 256]
    B = len(counts)
    q, kv = _kv_operands(B, Tq, S, H, hd, seed=100 + hd)
    k_len = torch.tensor(counts, dtype=torch.int32).cuda()
    with torch.no_grad():
        base = ops.small_attention_kv_cached(q, kv, H, k_len=k_len)
        # keys and values past each row's count overwritten with large finite values of both signs
        junk = kv.clone()
        g = torch.Generator().manual_seed(hd)
        for b, n in enumerate(counts):
            sign = torch.where(torch.rand(S - n, kv.shape[2], generator=g) < 0.5, -1.0, 1.0)
            junk[b, n:] = (sign * 3.0e38).to(BF16).cuda()
        assert torch.isfinite(junk.float()).all()
        assert torch.equal(ops.small_attention_kv_cached(q, junk, H, k_len=k_len), base)
        # other rows' counts change
        other = torch.tensor([300, 17, 1000, 513, 999], dtype=torch.int32).cuda()
        out2 = ops.small_attention_kv_cached(q, kv, H, k_len=other)
        assert torch.equal(out2[0], base[0]) and torch.equal(out2[3], base[3])
        # the empty chunks past a row's count are exact no-ops of the chunk-order merge: row 4 (256 keys, one chunk)
        # against a 256-key cache, where there is no other chunk at all
        short = ops.small_attention_kv_cached(q[4:5], kv[4:5, :256], H, k_len=k_len[4:5])
        assert torch.equal(short[0], base[4])
        assert torch.equal(ops.small_attention_kv_cached(q[4:5], kv[4:5, :256], H), base[4:5])
        # every row at S is the call without counts
        full = torch.full((B,), S, dtype=torch.int32).cuda()
        assert torch.equal(ops.small_attention_kv_cached(q, kv, H, k_len=full), ops.small_attention_kv_cached(q, kv, H))
    with pytest.raises(ops.FkError):
        ops.small_attention_kv_cached(q, kv, H, k_len=k_len.long())
    with pytest.raises(ops.FkError):
        ops.small_attention_kv_cached(q, kv, H, k_len=k_len[:3])
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# kernel: positions of a step whose rows sit at different positions
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,n_new,E,cap", [(5, 256, 256, 4096), (7, 48, 16, 128), (3, 100, 37, 1000), (1, 1, 1, 1)])
def test_stream_positions_match_torch(B, n_new, E, cap):
    from frankenstein_b200 import ops
    g = torch.Generator().manual_seed(B * n_new)
    lens = torch.randint(0, cap - n_new + 1, (B,), generator=g)
    lens[0] = 0
    lens[-1] = cap - n_new
    len_in = lens.to(torch.int32).cuda()
    len_out = torch.full((B,), -7, dtype=torch.int32).cuda()
    qid, qmin, qmax, pos, rows = ops.stream_positions(len_in, len_out, n_new, E, cap)
    p = lens[:, None] + torch.arange(n_new)[None]                     # [B, n_new]
    ref_qid = p // E
    assert torch.equal(qid.cpu(), ref_qid.to(torch.int32))
    assert torch.equal(pos.cpu(), p.to(torch.int32))
    assert torch.equal(rows.cpu(), (torch.arange(B)[:, None] * cap + p).reshape(-1))
    nt = (n_new + 63) // 64
    pad = torch.nn.functional.pad(ref_qid, (0, nt * 64 - n_new), value=-1).view(B, nt, 64)
    assert torch.equal(qmax.cpu(), pad.amax(-1).to(torch.int32))
    big = torch.nn.functional.pad(ref_qid, (0, nt * 64 - n_new), value=1 << 30).view(B, nt, 64)
    assert torch.equal(qmin.cpu(), big.amin(-1).to(torch.int32))
    assert torch.equal(len_out.cpu(), (lens + n_new).to(torch.int32))
    assert torch.equal(len_in.cpu(), lens.to(torch.int32))
    # the ranges are those of the general label-range kernel
    m = ops.LabelMask(qid)
    assert torch.equal(m.qmin, qmin) and torch.equal(m.qmax, qmax)


def test_stream_positions_rejects_without_launch():
    from frankenstein_b200 import _lib
    from frankenstein_b200._lib import lib, ptr, stream
    B, n = 3, 64
    a = torch.zeros(B, dtype=torch.int32, device="cuda")
    o = torch.zeros(B, dtype=torch.int32, device="cuda")
    i32 = torch.zeros(B * n, dtype=torch.int32, device="cuda")
    r64 = torch.zeros(B * n, dtype=torch.int64, device="cuda")

    def call(len_in=a, len_out=o, B=B, n_new=n, E=16, cap=128, rows=r64):
        return lib().fk_stream_positions(ptr(len_in), ptr(len_out), B, n_new, E, cap, ptr(i32), ptr(i32), ptr(i32), ptr(i32),
                                         ptr(rows), stream())
    torch.cuda.synchronize()
    before = _lib.launch_count()
    for bad in (dict(B=0), dict(B=65536), dict(n_new=0), dict(n_new=129), dict(E=0), dict(len_out=a), dict(len_in=None),
                dict(rows=None)):
        assert call(**bad) != 0, bad
    assert _lib.launch_count() == before
    assert call() == 0 and _lib.launch_count() == before + 1


# ------------------------------------------------------------------------------------------------
# Encoder.stream / BrainFormer.stream with staggered sessions
# ------------------------------------------------------------------------------------------------
STEPS = [1, 2, 1, 1, 1, 2, 1, 1, 1]                 # patches per step (every row advances by these)
RESETS = {2: [1], 4: [0], 5: [2]}                    # step -> rows reset before it: sessions of row 0 start at steps 0
                                                     # and 4 (reset mid-window), row 1 at 2, row 2 at 5


def _sessions(B, E, p, seed):
    """per row, the bins of its sessions: a list of [n_patches * p, E] tensors, consumed in order"""
    g = torch.Generator().manual_seed(seed)
    return [[torch.randn(16 * p, E, generator=g).cuda() for _ in range(3)] for _ in range(B)]


def _drive(stream, steps, resets, data, p, on_step):
    """feed every row its current session's next bins; before step i reset the rows in resets[i] (they move to their
    next session).  on_step(i, out, rows_state) with rows_state[r] = (session tensor, bins fed so far)."""
    B = len(data)
    sess, fed = [0] * B, [0] * B
    for i, n in enumerate(steps):
        for r in resets.get(i, []):
            sess[r] += 1
            fed[r] = 0
        if resets.get(i):
            stream.reset(resets[i])
        x = torch.stack([data[r][sess[r]][fed[r]:fed[r] + n * p] for r in range(B)])
        with pytest.MonkeyPatch.context() as m:
            _no_dense_attention(m)
            out = stream.step(x)
        for r in range(B):
            fed[r] += n * p
        on_step(i, out, [(data[r][sess[r]], fed[r]) for r in range(B)])


def _check_encoder(enc, steps, resets, seed, oracle_at=()):
    from oracle import brainformer_ref as o
    B, p, E = 3, enc.patch_size, enc.n_electrodes
    data = _sessions(B, E, p, seed)
    s = enc.stream(B)
    sd = {kk: vv.detach().float() for kk, vv in enc.state_dict().items()}
    cfg = dict(window_size=enc.config.window_size, patch_size=p, n_electrodes=E, head_dim=enc.config.head_dim,
               n_heads=enc.config.n_heads, rope_theta=enc.config.rope_theta)
    outs = []

    def on_step(i, y, state):
        n = steps[i] * E
        assert y.shape == (B, n, enc.config.dim) and y.dtype == torch.float32
        assert s.lengths == [fed // p * E for _, fed in state]
        for r, (x_r, fed) in enumerate(state):
            with torch.no_grad():
                off = enc(x_r[None, :fed])[0, -n:]
            rel_close(y[r], off, what=f"step {i} row {r} vs Encoder.forward")
            if i in oracle_at:
                with torch.no_grad():
                    ref = o.encoder_forward(sd, x_r[None, :fed].float(), cfg)[0, -n:]
                rel_close(y[r], ref, what=f"step {i} row {r} vs oracle")
        outs.append(y)
    _drive(s, steps, resets, data, p, on_step)
    return s, outs


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_encoder_staggered_sessions(hd):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(hd)
    enc = bf.Encoder(bf.MAEConfig(**_enc_cfg(hd))).cuda()
    s, _ = _check_encoder(enc, STEPS, RESETS, seed=hd, oracle_at={3, 8})
    with pytest.raises(bf.ops.FkError, match="lengths"):
        s.length
    assert _counters_zero()


def test_encoder_staggered_sessions_cfg2():
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(2)
    enc = bf.Encoder(bf.MAEConfig(**CFG2)).cuda()
    _check_encoder(enc, STEPS, RESETS, seed=2, oracle_at={6})
    assert _counters_zero()


# row 1's session: identical data and resets in both streams (its first reset, before step 0, puts both streams on the
# per-row path from the first step); rows 0 and 2 differ in data and schedule
IND_STEPS = [1, 2, 1, 1, 1, 2, 1]
IND_A = {0: [1], 3: [0, 1], 5: [2]}
IND_B = {0: [1, 2], 1: [0], 3: [1], 4: [2, 0]}


def _row_outputs(stream, resets, data, p, row):
    got = []
    _drive(stream, IND_STEPS, resets, data, p, lambda i, y, st: got.append(y[row].clone()))
    return got


@pytest.mark.parametrize("hd", [16, 64])
def test_encoder_row_independent_of_other_rows(hd):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(hd + 1)
    enc = bf.Encoder(bf.MAEConfig(**_enc_cfg(hd))).cuda()
    p, E = enc.patch_size, enc.n_electrodes
    da, db = _sessions(3, E, p, seed=1), _sessions(3, E, p, seed=2)
    db[1] = da[1]
    a = _row_outputs(enc.stream(3), IND_A, da, p, 1)
    b = _row_outputs(enc.stream(3), IND_B, db, p, 1)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert _counters_zero()


def _brainformer(hd, seed):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(seed)
    per = dict(n_output_tokens=8, output_dim=24, dim=128, n_layers=2, head_dim=16, hidden_dim=256, n_heads=8, n_kv_heads=8)
    model = bf.BrainFormer(bf.Config(encoder=bf.MAEConfig(**_enc_cfg(hd)), **per)).cuda()
    with torch.no_grad():
        model.learnable_queries.normal_()
    return model


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_brainformer_staggered_sessions(hd):
    model = _brainformer(hd, seed=11 + hd)
    enc = model.encoder
    p, E = enc.patch_size, enc.n_electrodes
    data = _sessions(3, E, p, seed=hd)
    s = model.stream(3)

    def on_step(i, pred, state):
        assert pred.shape == (3, 8, 24) and not pred.requires_grad
        assert s.lengths == [fed // p * E for _, fed in state]
        for r, (x_r, fed) in enumerate(state):
            with torch.no_grad():
                _, ref = model(x_r[None, :fed])
            rel_close(pred[r], ref[0], what=f"step {i} row {r} pred")
    _drive(s, STEPS, RESETS, data, p, on_step)
    # independence of row 1's pred from the other rows
    db = _sessions(3, E, p, seed=hd + 50)
    db[1] = data[1]
    a = _row_outputs(model.stream(3), IND_A, data, p, 1)
    b = _row_outputs(model.stream(3), IND_B, db, p, 1)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert _counters_zero()


def test_stream_rejections_leave_state():
    """bad rows, a step past the window for one row and bad shapes raise and change nothing; the next step is right"""
    from frankenstein_b200 import brainformer as bf
    model = _brainformer(32, seed=5)
    enc = model.encoder
    p, E = enc.patch_size, enc.n_electrodes
    data = _sessions(3, E, p, seed=9)
    s = model.stream(3)
    es = s.encoder_stream
    feed = lambda r, a, b: data[r][0][a * p:b * p]
    s.step(torch.stack([feed(r, 0, 3) for r in range(3)]))
    s.reset([1])
    s.step(torch.stack([feed(0, 3, 6), data[1][1][:3 * p], feed(2, 3, 6)]))
    assert s.lengths == [6 * E, 3 * E, 6 * E]
    snap = ([c.clone() for c in es.caches], [k.clone() for k in s.kv], es._len_dev.clone(), es._cur)
    for bad in ([3], [0, 0], [-1]):
        with pytest.raises(bf.ops.FkError):
            s.reset(bad)
    for x in (torch.zeros(3, 3 * p, E, device="cuda"),          # 6 + 3 patches: rows 0 and 2 past the 8-patch window
              torch.zeros(3, p + 1, E, device="cuda"),          # partial patch
              torch.zeros(2, p, E, device="cuda"),              # batch
              torch.zeros(3, p, E - 1, device="cuda")):         # electrodes
        with pytest.raises(bf.ops.FkError):
            s.step(x)
    torch.cuda.synchronize()
    assert s.lengths == [6 * E, 3 * E, 6 * E]
    assert all(torch.equal(a, b) for a, b in zip(snap[0], es.caches)) and all(torch.equal(a, b) for a, b in zip(snap[1], s.kv))
    assert torch.equal(snap[2], es._len_dev) and snap[3] == es._cur
    with pytest.raises(bf.ops.FkError, match="lengths"):
        s.length
    pred = s.step(torch.stack([feed(0, 6, 8), data[1][1][3 * p:5 * p], feed(2, 6, 8)]))
    for r, x_r in enumerate((data[0][0][:8 * p], data[1][1][:5 * p], data[2][0][:8 * p])):
        with torch.no_grad():
            _, ref = model(x_r[None])
        rel_close(pred[r], ref[0], what=f"row {r} after rejections")
    assert _counters_zero()


def test_lockstep_makes_no_per_row_launches():
    """a stream never reset row by row runs the lockstep path: no positions kernel, no per-row key counts"""
    from torch.profiler import ProfilerActivity, profile
    from frankenstein_b200 import ops
    model = _brainformer(32, seed=3)
    p, E = model.encoder.patch_size, model.encoder.n_electrodes
    x = torch.randn(2, 8 * p, E).cuda()
    calls = []
    orig = ops.small_attention_kv_cached

    def spy(*a, **k):
        calls.append(k.get("k_len"))
        return orig(*a, **k)
    s = model.stream(2)
    with pytest.MonkeyPatch.context() as m:
        m.setattr(ops, "small_attention_kv_cached", spy)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            s.step(x[:, :p])
            s.step(x[:, p:3 * p])
            s.reset()
            s.step(x[:, :2 * p])
            torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names and not any("stream_positions" in n for n in names)
    assert calls and all(k is None for k in calls)
    # after a per-row reset the positions kernel runs once per step and the perceiver gets the row counts
    s.reset([0])
    with pytest.MonkeyPatch.context() as m:
        m.setattr(ops, "small_attention_kv_cached", spy)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            s.step(x[:, :p])
            torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert sum("stream_positions" in n for n in names) == 1
    assert calls[-1] is not None
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# SoundStream.stream
# ------------------------------------------------------------------------------------------------
def _token_stream_feats(s, x, monkeypatch):
    """one step -> (indices, quantized, encoder features [B, n, D]) (features captured where the quantizer reads them)"""
    from frankenstein_b200 import vq_brain
    got = []
    orig = vq_brain.prepare_input

    def spy(e, cosine):
        got.append(e.clone())
        return orig(e, cosine)
    with monkeypatch.context() as m:
        m.setattr(vq_brain, "prepare_input", spy)
        ind, q = s.step(x)
    return ind, q, got[0].view(x.shape[0], x.shape[1] // 4, -1)


@pytest.mark.parametrize("cosine", [False, True])
def test_tokenizer_reset_rows(cosine, monkeypatch):
    from frankenstein_b200.ops import FkError
    from tests.test_tokenizer_stream_gpu import _check_tokens, _model, _signal
    m = _model(64, cosine)
    E = m.encoder.layers[0].in_channels
    B, T1, T2 = 3, 256, 512
    x = _signal(B, T1 + T2, E, seed=31 + cosine).cuda()
    fresh_bins = _signal(B, T2, E, seed=77).cuda()
    steps = [32, 4, 60, 12, 128, 20]                          # T1 = 256 bins, then T2 = 512 in the same steps twice
    s, plain, fresh = m.stream(B), m.stream(B), m.stream(B)   # s: row 1 reset after T1; plain: no reset
    t = 0
    for n in steps:
        for st in (s, plain):
            _token_stream_feats(st, x[:, t:t + n], monkeypatch)
        t += n
    s.reset([1])
    assert s.lengths == [T1, 0, T1]
    with pytest.raises(FkError, match="lengths"):
        s.length
    feats_s, feats_p, feats_f, ind_s = [], [], [], []
    t = 0
    for n in steps * 2:
        xs = x[:, T1 + t:T1 + t + n].clone()
        xs[1] = fresh_bins[1, t:t + n]
        a = _token_stream_feats(s, xs, monkeypatch)
        feats_s.append(a[2])
        ind_s.append((a[0], a[1]))
        feats_p.append(_token_stream_feats(plain, x[:, T1 + t:T1 + t + n], monkeypatch)[2])
        feats_f.append(_token_stream_feats(fresh, xs, monkeypatch)[2])
        t += n
    fs, fp, ff = (torch.cat(f, 1) for f in (feats_s, feats_p, feats_f))
    assert torch.equal(fs[1], ff[1]), "the reset row differs from a fresh stream"
    assert torch.equal(fs[0], fp[0]) and torch.equal(fs[2], fp[2]), "an untouched row changed"
    assert s.lengths == [T1 + T2, T2, T1 + T2]
    # tokens of every row against the offline eval path on that row's own session
    ind = torch.cat([i for i, _ in ind_s], 1)
    q = torch.cat([qq for _, qq in ind_s], 1)
    embed = m.quantizer.codebook
    for r, xr in enumerate((x[0], fresh_bins[1, :T2], x[2])):
        with torch.no_grad():
            ref_ind, ref_q = m.get_quantize_vectors(xr[None])
            feats = m.encoder(xr[None])
        n_tok = T2 // 4
        _check_tokens(ind[r:r + 1], q[r:r + 1], ref_ind[:, -n_tok:], ref_q[:, -n_tok:], feats[:, -n_tok:], embed, cosine,
                      f"cos {cosine} row {r}")
    for bad in ([3], [1, 1]):
        with pytest.raises(FkError):
            s.reset(bad)
    assert s.lengths == [T1 + T2, T2, T1 + T2]
    assert _counters_zero()
