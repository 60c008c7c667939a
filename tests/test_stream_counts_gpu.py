"""Streams whose rows receive different amounts of data in one step (`step(x, counts)`): the positions kernel and the
convolution row kernel with per-row counts against torch, Encoder / BrainFormer / SoundStream streams under an
asynchronous arrival schedule (counts 0, 1 or 2 patches, resets, rows waiting at the end of the window), each row against
the offline forward on its own bins, bit-for-bit independence of a row from the other rows, filler that never matters,
the unchanged lockstep path and rejections that change nothing.
"""
import random

import pytest
import torch

from tests.test_encoder_stream_gpu import CFG2, _counters_zero, _enc_cfg, _no_dense_attention, rel_close
from tests.test_stream_sessions_gpu import _brainformer
from tests.test_tokenizer_stream_gpu import _check_tokens, _model, _signal

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
NO_LABEL = -2 ** 31


# ------------------------------------------------------------------------------------------------
# kernels
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,n_new,E,cap", [(6, 256, 256, 4096), (7, 48, 16, 128), (5, 100, 37, 1000)])
def test_stream_positions_counts_match_torch(B, n_new, E, cap):
    from frankenstein_b200 import ops
    g = torch.Generator().manual_seed(B * n_new + 1)
    counts = torch.randint(0, n_new + 1, (B,), generator=g)
    counts[0], counts[1], counts[2] = 0, n_new, 1
    lens = (torch.rand(B, generator=g) * (cap - counts + 1).double()).long()
    lens[1] = cap - n_new                                   # count = n_new that ends exactly at the window
    lens[0] = cap                                           # a row at the end of the window, count 0
    len_in = lens.to(torch.int32).cuda()
    len_out = torch.full((B,), -7, dtype=torch.int32).cuda()
    cnt = counts.to(torch.int32).cuda()
    qid, qmin, qmax, pos, rows = ops.stream_positions(len_in, len_out, n_new, E, cap, cnt)
    i = torch.arange(n_new)[None]
    p = lens[:, None] + i
    live = i < counts[:, None]
    ref_qid = torch.where(live, p // E, NO_LABEL)
    assert torch.equal(qid.cpu(), ref_qid.to(torch.int32))
    assert torch.equal(pos.cpu(), p.clamp(max=cap - 1).to(torch.int32))
    ref_rows = torch.where(live, torch.arange(B)[:, None] * cap + p, B * cap)
    assert torch.equal(rows.cpu(), ref_rows.reshape(-1))
    assert bool((rows.cpu()[live.reshape(-1)] < B * cap).all())
    nt = (n_new + 63) // 64
    hi = torch.nn.functional.pad(ref_qid, (0, nt * 64 - n_new), value=NO_LABEL).view(B, nt, 64)
    lo = torch.nn.functional.pad(ref_qid, (0, nt * 64 - n_new), value=1 << 30).view(B, nt, 64)
    assert torch.equal(qmax.cpu(), hi.amax(-1).to(torch.int32))
    assert torch.equal(qmin.cpu(), lo.amin(-1).to(torch.int32))
    m = ops.LabelMask(qid)                                  # the ranges of the general label-range kernel
    assert torch.equal(m.qmin, qmin) and torch.equal(m.qmax, qmax)
    assert torch.equal(len_out.cpu(), (lens + counts).to(torch.int32))
    # NULL counts: the entry point without counts, bit for bit
    len_in2 = torch.clamp(lens, max=cap - n_new).to(torch.int32).cuda()
    a = ops.stream_positions(len_in2, len_out, n_new, E, cap)
    o2 = torch.empty_like(len_out)
    from frankenstein_b200._lib import lib, ptr, stream
    b_ = [torch.empty_like(t) for t in a]
    assert lib().fk_stream_positions(ptr(len_in2), ptr(o2), B, n_new, E, cap, *(ptr(t) for t in b_), stream()) == 0
    assert all(torch.equal(x, y) for x, y in zip(a, b_)) and torch.equal(o2, len_out)
    full = torch.full((B,), n_new, dtype=torch.int32).cuda()
    assert all(torch.equal(x, y) for x, y in zip(a, ops.stream_positions(len_in2, o2, n_new, E, cap, full)))


def _launch_rows_counts(x, r, elu, hist_in, hist_out, counts, rpt, total, C):
    from frankenstein_b200 import conv
    from frankenstein_b200._lib import lib, ptr, stream
    B, n, _ = x.shape
    h = 0 if hist_in is None else hist_in.shape[1]
    out = torch.full((total, C), 7.0, device=x.device, dtype=BF16)              # every row must be written
    rs = (0, 0) if r is None else conv._row_strides(r)
    rc = lib().fk_conv_stream_rows_counts(ptr(x), 0 if x.dtype == torch.float32 else 1, *conv._row_strides(x), ptr(r), *rs,
                                          ptr(hist_in), ptr(hist_out), ptr(counts), B, n, h, C, int(elu), ptr(out), rpt,
                                          total, stream())
    return rc, out


@pytest.mark.parametrize("dtype", [torch.float32, BF16])
@pytest.mark.parametrize("res,elu", [(False, False), (True, True), (False, True)])
@pytest.mark.parametrize("h", [0, 1, 3, 6])
def test_stream_rows_counts_match_torch(dtype, res, elu, h):
    B, n, C = 5, 8, 64
    cnt = [0, n, 3, 1, 6]
    g = torch.Generator().manual_seed(h * 7 + res + 2 * elu)
    x = (torch.randn(B, n, C, generator=g) * 3).cuda().to(dtype)
    r = (torch.randn(B, n, C, generator=g) * 2).cuda().to(BF16) if res else None
    for b, c in enumerate(cnt):                              # filler past each count is never read
        x[b, c:] = float("nan")
        if r is not None:
            r[b, c:] = float("nan")
    hist_in = torch.randn(B, h, C, generator=g).cuda().to(BF16) if h else None
    hist_out = torch.full((B, h, C), 5.0, device="cuda", dtype=BF16) if h else None
    rpt = n + h + 1
    total = B * rpt + h + 1
    counts = torch.tensor(cnt, dtype=torch.int32).cuda()
    rc, out = _launch_rows_counts(x, r, elu, hist_in, hist_out, counts, rpt, total, C)
    assert rc == 0
    ref = torch.zeros(total, C, device="cuda", dtype=BF16)
    for b, c in enumerate(cnt):
        s = x[b, :c] if r is None else (x[b, :c].float() + r[b, :c].float()).to(BF16)
        if elu:
            s = torch.nn.functional.elu(s)
        full = s.to(BF16) if hist_in is None else torch.cat([hist_in[b], s.to(BF16)], 0)
        ref[b * rpt:b * rpt + full.shape[0]] = full
        if h:
            assert torch.equal(hist_out[b].view(torch.int16), full[full.shape[0] - h:].view(torch.int16)), f"history {b}"
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))
    if h:
        assert torch.equal(hist_out[0], hist_in[0])              # count 0 carries the history over bit for bit
    # full counts == NULL counts == the entry point without counts
    xf = torch.randn(B, n, C, generator=g).cuda().to(dtype)
    hof = torch.zeros_like(hist_out) if h else None
    full = torch.full((B,), n, dtype=torch.int32).cuda()
    a = _launch_rows_counts(xf, None, elu, hist_in, hist_out, full, rpt, total, C)[1]
    b_ = _launch_rows_counts(xf, None, elu, hist_in, hof, None, rpt, total, C)[1]
    from tests.test_tokenizer_stream_gpu import _launch_rows
    c_ = _launch_rows(xf, None, elu, hist_in, hof, rpt, total, C)[1]
    assert torch.equal(a, b_) and torch.equal(a, c_)
    if h:
        assert torch.equal(hist_out, hof)


# ------------------------------------------------------------------------------------------------
# asynchronous arrival: Encoder / BrainFormer
# ------------------------------------------------------------------------------------------------
def schedule(B, W, n_steps, seed):
    """[(resets, counts)] per step: counts in {0, 1, 2} patches within the window of W patches, one row idle each step
    (so every step takes the per-row path), rows at the end of the window wait there (count 0) until a reset"""
    rng = random.Random(seed)
    fed = [0] * B
    out = []
    for i in range(n_steps):
        resets = [r for r in range(B) if (fed[r] == W and rng.random() < 0.4) or (fed[r] and rng.random() < 0.03)]
        for r in resets:
            fed[r] = 0
        counts = [min(rng.choice([0, 1, 2, 2, 2]), W - fed[r]) for r in range(B)]
        counts[i % B] = 0
        for r in range(B):
            fed[r] += counts[r]
        out.append((resets, counts))
    return out


def _fill(shape, filler, g):
    if filler == "zero":
        return torch.zeros(shape)
    if filler == "nan":
        return torch.full(shape, float("nan"))
    return torch.where(torch.rand(shape, generator=g) < 0.5, -3.0e38, 3.0e38)


def _drive(stream, enc, sched, seed, on_step, filler="zero", data_seed=None):
    """feed the schedule: each row its current session's next counts[r] patches, filler after them; a reset starts a new
    session.  on_step(i, out, counts, [(session bins, patches fed)])"""
    p, E = enc.patch_size, enc.n_electrodes
    W = enc.block_size // E
    g = torch.Generator().manual_seed(seed if data_seed is None else data_seed)
    gf = torch.Generator().manual_seed(12345)
    B = len(sched[0][1])
    sess = [torch.randn(W * p, E, generator=g).cuda() for _ in range(B)]
    fed = [0] * B
    for i, (resets, counts) in enumerate(sched):
        if resets:
            stream.reset(resets)
            for r in resets:
                sess[r], fed[r] = torch.randn(W * p, E, generator=g).cuda(), 0
        x = _fill((B, 2 * p, E), filler, gf).cuda()
        for r in range(B):
            x[r, :counts[r] * p] = sess[r][fed[r] * p:(fed[r] + counts[r]) * p]
        with pytest.MonkeyPatch.context() as m:
            _no_dense_attention(m)
            out = stream.step(x, counts)
        for r in range(B):
            fed[r] += counts[r]
        on_step(i, out, counts, [(sess[r], fed[r]) for r in range(B)])


def _check_encoder_async(enc, B, n_steps, seed, oracle_at=()):
    from oracle import brainformer_ref as o
    p, E = enc.patch_size, enc.n_electrodes
    W = enc.block_size // E
    sched = schedule(B, W, n_steps, seed)
    s = enc.stream(B)
    sd = {kk: vv.detach().float() for kk, vv in enc.state_dict().items()}
    cfg = dict(window_size=enc.config.window_size, patch_size=p, n_electrodes=E, head_dim=enc.config.head_dim,
               n_heads=enc.config.n_heads, rope_theta=enc.config.rope_theta)
    at_end = [0]

    def on_step(i, y, counts, state):
        assert y.shape == (B, 2 * E, enc.config.dim) and y.dtype == torch.float32
        assert s.lengths == [fed * E for _, fed in state]
        for r, (x_r, fed) in enumerate(state):
            n = counts[r] * E
            assert bool((y[r, n:] == 0).all()), f"step {i} row {r}: slots past the count are not zero"
            at_end[0] += fed == W and counts[r] == 0
            if n == 0:
                continue
            with torch.no_grad():
                off = enc(x_r[None, :fed * p])[0, -n:]
            rel_close(y[r, :n], off, what=f"step {i} row {r} vs Encoder.forward")
            if i in oracle_at:
                with torch.no_grad():
                    ref = o.encoder_forward(sd, x_r[None, :fed * p].float(), cfg)[0, -n:]
                rel_close(y[r, :n], ref, what=f"step {i} row {r} vs oracle")
    _drive(s, enc, sched, seed, on_step)
    assert at_end[0] > 0, "no row waited at the end of its window"
    return s


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_encoder_async_counts(hd):
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(hd)
    enc = bf.Encoder(bf.MAEConfig(**_enc_cfg(hd))).cuda()
    _check_encoder_async(enc, 4, 16, seed=hd, oracle_at={5, 11})
    assert _counters_zero()


def test_encoder_async_counts_cfg2():
    from frankenstein_b200 import brainformer as bf
    torch.manual_seed(2)
    enc = bf.Encoder(bf.MAEConfig(**CFG2)).cuda()
    _check_encoder_async(enc, 3, 24, seed=3, oracle_at={9})
    assert _counters_zero()


@pytest.mark.parametrize("hd", [16, 32, 64])
def test_brainformer_async_counts(hd):
    model = _brainformer(hd, seed=21 + hd)
    enc = model.encoder
    p, E = enc.patch_size, enc.n_electrodes
    B = 4
    sched = schedule(B, enc.block_size // E, 14, seed=40 + hd)
    s = model.stream(B)
    prev = [None] * B

    def on_step(i, pred, counts, state):
        assert pred.shape == (B, 8, 24) and torch.isfinite(pred).all()
        for r, (x_r, fed) in enumerate(state):
            if r in sched[i][0] or fed == 0:
                prev[r] = None                                  # a new session; with no context yet the perceiver runs
            if fed == 0:                                        # over an empty context (finite, checked above)
                continue
            if counts[r] == 0 and prev[r] is not None:
                assert torch.equal(pred[r], prev[r]), f"step {i} row {r}: a count-0 row's prediction changed"
            with torch.no_grad():
                _, ref = model(x_r[None, :fed * p])
            rel_close(pred[r], ref[0], what=f"step {i} row {r} pred")
            prev[r] = pred[r].clone()
    _drive(s, enc, sched, 40 + hd, on_step)
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# row independence and filler
# ------------------------------------------------------------------------------------------------
def _outputs(stream, enc, sched, seed, filler="zero", data_seed=None):
    got = []
    _drive(stream, enc, sched, seed, lambda i, y, c, st: got.append(y.clone()), filler, data_seed)
    return got


@pytest.mark.parametrize("kind", ["encoder", "brainformer"])
def test_row_independent_of_other_rows(kind):
    """row 1: the same data, counts and resets in both streams; the other rows differ in data, counts and resets"""
    model = _brainformer(32, seed=8)
    enc = model.encoder
    W = enc.block_size // enc.n_electrodes
    a_s, b_s = schedule(3, W, 12, seed=1), schedule(3, W, 12, seed=2)
    for i in range(12):                                     # row 1 of b follows row 1 of a
        b_s[i][1][1] = a_s[i][1][1]
        b_s[i] = ([r for r in b_s[i][0] if r != 1] + [1] * (1 in a_s[i][0]), b_s[i][1])
    mk = (lambda: enc.stream(3)) if kind == "encoder" else (lambda: model.stream(3))

    # the data of row 1 must be the same: drive with a data generator per row via one seed, then patch row 1's data
    def run(sched, seed):
        got = []
        p, E = enc.patch_size, enc.n_electrodes
        g = torch.Generator().manual_seed(seed)
        g1 = torch.Generator().manual_seed(99)
        sess = [torch.randn(W * p, E, generator=g1 if r == 1 else g).cuda() for r in range(3)]
        fed = [0] * 3
        s = mk()
        for resets, counts in sched:
            if resets:
                s.reset(resets)
                for r in resets:
                    sess[r], fed[r] = torch.randn(W * p, E, generator=g1 if r == 1 else g).cuda(), 0
            x = torch.randn(3, 2 * p, E, generator=g).cuda()
            for r in range(3):
                x[r, :counts[r] * p] = sess[r][fed[r] * p:(fed[r] + counts[r]) * p]
                fed[r] += counts[r]
            x[1, counts[1] * p:] = 0
            got.append(s.step(x, counts)[1].clone())
        return got
    a, b = run(a_s, 1), run(b_s, 2)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert _counters_zero()


@pytest.mark.parametrize("kind", ["encoder", "brainformer"])
def test_filler_never_matters(kind):
    model = _brainformer(64, seed=9)
    enc = model.encoder
    sched = schedule(3, enc.block_size // enc.n_electrodes, 12, seed=5)
    res = {}
    for filler in ("zero", "nan", "big"):
        s = enc.stream(3) if kind == "encoder" else model.stream(3)
        res[filler] = _outputs(s, enc, sched, 5, filler)
        es = s if kind == "encoder" else s.encoder_stream
        assert all(bool(torch.isfinite(c.float()).all()) for c in es.caches), filler
        if kind != "encoder":
            assert all(bool(torch.isfinite(k.float()).all()) for k in s.kv), filler
    for filler in ("nan", "big"):
        assert all(torch.equal(x, y) for x, y in zip(res["zero"], res[filler])), filler
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# the unchanged path, all-zero steps, rejections
# ------------------------------------------------------------------------------------------------
def _cuda_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_full_counts_are_the_plain_step():
    model = _brainformer(32, seed=4)
    p, E = model.encoder.patch_size, model.encoder.n_electrodes
    x = torch.randn(3, 8 * p, E).cuda()
    plan = [(0, 1), (1, 3), (3, 4), (4, 6)]
    for mk in (lambda: model.encoder.stream(3), lambda: model.stream(3)):
        runs = []
        for counts in ("warm-up", "plain", None, "full"):       # (first calls do one-time work: the warm-up)
            s = mk()
            outs, names = [], []
            for j, (a, b) in enumerate(plan):
                if j == 2:
                    s.reset([1])                              # the per-row path from here on
                arg = () if counts in ("plain", "warm-up") else ((None,) if counts is None else ([b - a] * 3,))
                o, nm = _cuda_names(lambda: s.step(x[:, a * p:b * p], *arg))
                outs.append(o)
                names.append(nm)
            runs.append((outs, names))
        runs = runs[1:]
        for outs, names in runs[1:]:
            assert all(torch.equal(u, v) for u, v in zip(outs, runs[0][0]))
            assert names == runs[0][1]
    m = _model(64, False)
    xt = _signal(2, T=64, C=64, seed=1).cuda()
    runs = []
    for counts in ("warm-up", "plain", None, "full"):
        s = m.stream(2, reconstruct=True)
        outs, names = [], []
        for a, b in ((0, 16), (16, 24), (24, 64)):
            arg = () if counts in ("plain", "warm-up") else ((None,) if counts is None else ([b - a] * 2,))
            o, nm = _cuda_names(lambda: s.step(xt[:, a:b], *arg))
            outs.extend(o)
            names.append(nm)
        runs.append((outs, names))
    runs = runs[1:]
    for outs, names in runs[1:]:
        assert all(torch.equal(u, v) for u, v in zip(outs, runs[0][0]))
        assert names == runs[0][1]
    assert _counters_zero()


def test_all_zero_counts_change_nothing():
    model = _brainformer(16, seed=6)
    p, E = model.encoder.patch_size, model.encoder.n_electrodes
    x = torch.randn(3, 4 * p, E).cuda()
    s = model.stream(3)
    es = s.encoder_stream
    pred0 = s.step(x[:, :2 * p], [2, 1, 0])
    snap = ([c.clone() for c in es.caches], [k.clone() for k in s.kv], es._len_dev[es._cur].clone(), s.lengths)
    pred1 = s.step(torch.full((3, 2 * p, E), float("nan")).cuda(), [0, 0, 0])
    assert torch.equal(pred1[:2], pred0[:2]) and torch.isfinite(pred1[2]).all()
    assert s.lengths == snap[3] and torch.equal(es._len_dev[es._cur], snap[2])
    assert all(torch.equal(a, b) for a, b in zip(snap[0], es.caches)) and all(torch.equal(a, b) for a, b in zip(snap[1], s.kv))
    y = es.step(torch.randn(3, p, E).cuda(), [0, 0, 0])
    assert bool((y == 0).all()) and s.lengths == snap[3]
    # a row at the end of the window with count 0 does not hold up the others
    s2 = model.encoder.stream(2)
    W = model.encoder.block_size // E
    for _ in range(W // 2):
        s2.step(torch.randn(2, 2 * p, E).cuda(), [2, 0])
    assert s2.lengths == [W * E, 0]
    s2.step(torch.randn(2, 2 * p, E).cuda(), [0, 2])
    assert s2.lengths == [W * E, 2 * E]
    assert _counters_zero()


def test_count_rejections_change_nothing():
    from frankenstein_b200 import _lib, ops
    model = _brainformer(32, seed=7)
    p, E = model.encoder.patch_size, model.encoder.n_electrodes
    W = model.encoder.block_size // E
    s = model.stream(3)
    es = s.encoder_stream
    s.step(torch.randn(3, W * p, E).cuda()[:, :2 * p], [2, 1, 0])
    for _ in range(W // 2 - 1):
        s.step(torch.randn(3, 2 * p, E).cuda(), [2, 0, 1])
    assert s.lengths == [W * E, E, (W // 2 - 1) * E]
    torch.cuda.synchronize()
    snap = ([c.clone() for c in es.caches], [k.clone() for k in s.kv], es._len_dev.clone(), es._cur, s.lengths)
    before = _lib.launch_count()
    x = torch.randn(3, 2 * p, E).cuda()
    for bad, match in (([1, 1], "2 counts"), ([1, 1, 1, 1], "4 counts"), ([0, -1, 0], r"rows \[1\]"),
                       ([0, 3, 0], r"rows \[1\]"), ([1, 0, 2], r"rows \[0\]"), ([0, 1.0, 0], "ints"), (5, "ints")):
        with pytest.raises(ops.FkError, match=match):
            s.step(x, bad)
    assert _lib.launch_count() == before
    torch.cuda.synchronize()
    assert s.lengths == snap[4] and torch.equal(es._len_dev, snap[2]) and es._cur == snap[3]
    assert all(torch.equal(a, b) for a, b in zip(snap[0], es.caches)) and all(torch.equal(a, b) for a, b in zip(snap[1], s.kv))
    # tokenizer
    m = _model(64, True)
    t = m.stream(3, reconstruct=True)
    xt = _signal(3, T=32, C=64, seed=2).cuda()
    t.step(xt, [32, 8, 0])
    hist = [[L.hist.clone() for L in layers if L.hist is not None] for layers in t._layers]
    before = _lib.launch_count()
    for bad, match in (([4, 4], "2 counts"), ([4, -4, 4], r"rows \[1\]"), ([36, 4, 4], r"rows \[0\]"),
                       ([4, 6, 2], r"rows \[1, 2\]")):
        with pytest.raises(ops.FkError, match=match):
            t.step(xt, bad)
    assert _lib.launch_count() == before and t.lengths == [32, 8, 0] and t._cur == 1
    now = [[L.hist for L in layers if L.hist is not None] for layers in t._layers]
    assert all(torch.equal(a, b) for ha, hb in zip(hist, now) for a, b in zip(ha, hb))
    assert _counters_zero()


# ------------------------------------------------------------------------------------------------
# SoundStream.stream
# ------------------------------------------------------------------------------------------------
def _tok_schedule(B, n_steps, T, seed):
    rng = random.Random(seed)
    return [[rng.choice([0, 4, 8, T // 2, T]) if (i + r) % 3 else 0 for r in range(B)] for i in range(n_steps)]


def _drive_tokens(s, rows, sched, T, filler, monkeypatch):
    """feed rows[r] (bins [N, E]) by the schedule; returns per row (indices, quantized, features, decoder bins) of its own
    new slots, concatenated"""
    from frankenstein_b200 import vq_brain
    B = len(rows)
    E = rows[0].shape[1]
    gf = torch.Generator().manual_seed(3)
    fed = [0] * B
    got = [[[], [], [], []] for _ in range(B)]
    for counts in sched:
        x = _fill((B, T, E), filler, gf).cuda()
        for r in range(B):
            x[r, :counts[r]] = rows[r][fed[r]:fed[r] + counts[r]]
        feats = []
        orig = vq_brain.prepare_input

        def spy(e, cosine):
            feats.append(e.clone())
            return orig(e, cosine)
        with monkeypatch.context() as mp:
            mp.setattr(vq_brain, "prepare_input", spy)
            out = s.step(x, counts)
        f = feats[0].view(B, T // 4, -1)
        for r in range(B):
            n = counts[r] // 4
            assert bool((out[0][r, n:] == -1).all()) and bool((out[1][r, n:] == 0).all())
            got[r][0].append(out[0][r, :n])
            got[r][1].append(out[1][r, :n])
            got[r][2].append(f[r, :n])
            if len(out) == 3:
                assert bool((out[2][r, counts[r]:] == 0).all())
                got[r][3].append(out[2][r, :counts[r]])
            fed[r] += counts[r]
    assert s.lengths == fed
    return [[torch.cat(v, 0) for v in g if v] for g in got], fed


@pytest.mark.parametrize("B", [1, 2, 3])
@pytest.mark.parametrize("cosine", [False, True])
def test_tokenizer_counts_match_offline(B, cosine, monkeypatch):
    m = _model(64, cosine)
    T = 32
    sched = _tok_schedule(B, 40, T, seed=B + 10 * cosine)
    total = max(sum(c[r] for c in sched) for r in range(B))
    rows = _signal(B, total, 64, seed=17 + B).cuda()
    s = m.stream(B, reconstruct=True)
    got, fed = _drive_tokens(s, [rows[r] for r in range(B)], sched, T, "zero", monkeypatch)
    embed = m.quantizer.codebook
    for r in range(B):
        x_r = rows[r:r + 1, :fed[r]]
        ind, q, feats, o = got[r]
        with torch.no_grad():
            ref_ind, ref_q = m.get_quantize_vectors(x_r)
            ref_feats = m.encoder(x_r)
            ref_o = m.decoder(q[None])
        assert torch.equal(feats, ref_feats[0]), f"row {r}: encoder features differ from Encoder.forward"
        _check_tokens(ind[None], q[None], ref_ind, ref_q, ref_feats, embed, cosine, f"B {B} cos {cosine} row {r}")
        print(f"B {B} row {r}: decoder bit-equal to Decoder.forward: {torch.equal(o, ref_o[0])}")
        rel_close(o, ref_o[0], rtol=1e-2, what=f"row {r} decoder")
    assert _counters_zero()


def test_tokenizer_filler_and_idle_histories(monkeypatch):
    m = _model(64, False)
    B, T = 3, 32
    sched = _tok_schedule(B, 20, T, seed=4)
    total = max(sum(c[r] for c in sched) for r in range(B))
    rows = _signal(B, total, 64, seed=5).cuda()
    res = {}
    for filler in ("zero", "nan", "big"):
        s = m.stream(B, reconstruct=True)
        res[filler] = _drive_tokens(s, [rows[r] for r in range(B)], sched, T, filler, monkeypatch)[0]
        for layers in s._layers:
            for L in layers:
                if L.hist is not None:
                    assert bool(torch.isfinite(L.hist.float()).all()), filler
    for filler in ("nan", "big"):
        assert all(torch.equal(a, b) for ra, rb in zip(res["zero"], res[filler]) for a, b in zip(ra, rb)), filler
    # a count-0 row keeps every history bit for bit, the others move on
    s = m.stream(B, reconstruct=True)
    s.step(rows[:, :T], [T, 8, 4])
    snap = [[L.hist[s._cur].clone() for L in layers if L.hist is not None] for layers in s._layers]
    out = s.step(torch.full((B, T, 64), float("nan")).cuda(), [0, 0, 0])
    assert bool((out[0] == -1).all()) and bool((out[1] == 0).all()) and bool((out[2] == 0).all())
    now = [[L.hist[s._cur] for L in layers if L.hist is not None] for layers in s._layers]
    assert all(torch.equal(a, b) for ha, hb in zip(snap, now) for a, b in zip(ha, hb))
    s.step(rows[:, T:2 * T], [0, T, 0])
    now = [[L.hist[s._cur] for L in layers if L.hist is not None] for layers in s._layers]
    assert all(torch.equal(a[0], b[0]) and torch.equal(a[2], b[2]) for ha, hb in zip(snap, now) for a, b in zip(ha, hb))
    assert s.lengths == [T, 8 + T, 4]
    assert _counters_zero()
