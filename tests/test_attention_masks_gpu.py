"""Self-attention kernels (attention_tc.cu, and the mma.sync cross-check kernels of attention.cu) against a float64
reference computed from the kernels' exact bf16 operands, under arbitrary label masks.

Visibility rule: key j is visible to query i  <=>  kid[b, j] <= qid[b, i], for every int32 label.  Every check is per
row (or per tensor for the key gradients), never against the largest element of the whole output:
  out   per-row max error / the largest |v| among that row's visible keys       <= OUT_TOL
  lse   absolute error, log2 units                                              <= LSE_TOL
  grads relative Frobenius error per tensor, and per row for dq                 <= GRAD_TOL
  rows with no visible key: exact zeros in out and dq, lse = +inf;  keys visible to no query: exact zeros in dk / dv.
The comparator itself is tested without a GPU (test_comparator_rejects_one_key): it must reject a reference with one
key more or one key less and an lse that counts one extra key.
"""
import math

import pytest
import torch

I32MAX, I32MIN = 2 ** 31 - 1, -2 ** 31
LOG2E = 1.0 / math.log(2.0)

# Largest errors over every case of this file on a B200 (1000 W): out 4.2e-3, lse 3.3e-6 (3.1e-5 with logits of std 30),
# dq / dk / dv 3.6e-3 / 3.4e-3 / 2.5e-3 (6.7e-3 / 6.4e-3 / 1.8e-3 with logits of std 30), dq per row 4.3e-2 (9.4e-2).
OUT_TOL = 8e-3          # bf16 rounding of O and of P: ~2^-9 of |v|
LSE_TOL = 1e-4          # one extra key of a 4096-key row moves lse by 3.5e-4
GRAD_TOL = 1e-2
DQ_ROW_TOL = 0.1        # per row, against max(|row|, rms row): a row's dS carries the bf16 rounding of its O in delta

PATHS = {
    "tc": {},
    "tc-staged": {"ATTN_BWD_STATS": "staged"},
    "tc-transposed": {"ATTN_BWD_OPERANDS": "transposed"},
    "legacy": {"ATTN_FWD_IMPL": "legacy", "ATTN_BWD_IMPL": "legacy"},
}
KINDS = ["causal", "anticausal", "random", "independent", "leftpad", "late", "empty_rows", "all_but_last",
         "extremes", "block7", "block48", "block64", "block256", "gathered", "padding"]
SHAPES = [1, 63, 65, 127, 129, 300, 513, 1000]


# ------------------------------------------------------------------------------------------------
# labels
# ------------------------------------------------------------------------------------------------
def make_labels(kind, B, S, g):
    """(qid, kid) int64 CPU tensors [B, S] for one mask family; None for no mask."""
    ar = torch.arange(S).expand(B, S)
    if kind == "none":
        return None
    if kind == "causal":                                  # token-level causal: row 0 sees exactly key 0
        return ar.clone(), ar.clone()
    if kind == "anticausal":                              # row S-1 sees exactly key S-1 (in the ragged tail)
        return -ar, -ar
    if kind == "random":                                  # unsorted labels, qid == kid
        ids = torch.randint(0, max(S // 8, 2), (B, S), generator=g)
        return ids, ids.clone()
    if kind == "independent":
        return torch.randint(0, 16, (B, S), generator=g), torch.randint(0, 16, (B, S), generator=g)
    if kind in ("leftpad", "padding"):                    # LabelMask.padding: padded keys INT32_MAX, padded queries -1
        pad = torch.zeros(B, S, dtype=torch.bool)
        for b in range(B):
            n = min(S, 17 * (b + 1) + S // 5)
            if kind == "leftpad":
                pad[b, :n] = True
            else:
                pad[b, S - n:] = True
        return torch.where(pad, -1, 0), torch.where(pad, I32MAX, 0)
    if kind == "late":
        # keys before `start` carry label 1, later ones 0; rows labelled 0 first see a key >= 2 key tiles in, after
        # tiles that the rows labelled 1 of the same work item need
        start = min(2 * 128 + 37, S // 2)
        kid = torch.where(ar >= start, 0, 1)
        return torch.randint(0, 2, (B, S), generator=g), kid
    if kind == "empty_rows":                              # block causal with scattered queries that see nothing
        kid = ar // 16
        qid = kid.clone()
        qid[torch.rand(B, S, generator=g) < 0.1] = -1
        return qid, kid
    if kind == "all_but_last":
        kid = torch.zeros(B, S, dtype=torch.long)
        kid[:, -1] = 1
        return torch.zeros(B, S, dtype=torch.long), kid
    if kind == "int32max":                                # every query sees every key
        return torch.full((B, S), I32MAX), torch.randint(I32MIN, I32MAX, (B, S), generator=g)
    if kind == "extremes":
        kv = torch.tensor([I32MIN, I32MIN + 1, -3, 0, 5, I32MAX - 1, I32MAX])
        qv = torch.tensor([I32MIN, I32MIN + 1, 0, 5, I32MAX - 1, I32MAX])
        return (qv[torch.randint(0, len(qv), (B, S), generator=g)], kv[torch.randint(0, len(kv), (B, S), generator=g)])
    if kind.startswith("block"):
        ids = ar // int(kind[5:])
        return ids, ids.clone()
    if kind == "gathered":                                # sorted random subset of 4 S positions, 32 positions a block
        ids = torch.stack([torch.sort(torch.randperm(4 * S, generator=g)[:S])[0] for _ in range(B)]) // 32
        return ids, ids.clone()
    raise ValueError(kind)


def visibility(labels, B, S, device):
    """bool [B, 1, S, S]: LabelMask.dense() semantics."""
    if labels is None:
        return torch.ones(B, 1, S, S, dtype=torch.bool, device=device)
    qid, kid = (t.to(device) for t in labels)
    return kid[:, None, None, :] <= qid[:, None, :, None]


# ------------------------------------------------------------------------------------------------
# float64 reference and comparator (device agnostic)
# ------------------------------------------------------------------------------------------------
def reference(q, k, v, vis, scale, d_o):
    """q / k / v / d_o: [B, S, H, hd] exact operands; vis [B, 1, S, S].  Returns float64 out [B, S, H, hd], lse [B, H, S]
    (log2 domain, +inf for empty rows), delta [B, H, S] and dq / dk / dv (gradients of sum(out * d_o))."""
    qd, kd, vd = (t.detach().double().requires_grad_(True) for t in (q, k, v))
    s = torch.einsum("bihd,bjhd->bhij", qd, kd) * scale
    s = s.masked_fill(~vis, -math.inf)
    m = s.detach().amax(-1, keepdim=True)
    m = torch.where(torch.isfinite(m), m, torch.zeros_like(m))
    p = torch.exp(s - m)
    l = p.sum(-1, keepdim=True)
    o = (p @ vd.transpose(1, 2)) / torch.where(l > 0, l, torch.ones_like(l))
    out = o.transpose(1, 2)
    (out * d_o.double()).sum().backward()
    lse = torch.where(l > 0, (m + torch.log(l)) * LOG2E, torch.full_like(l, math.inf)).squeeze(-1)
    delta = (out.detach() * d_o.double()).sum(-1).transpose(1, 2)
    return dict(out=out.detach(), lse=lse.detach(), delta=delta, dq=qd.grad, dk=kd.grad, dv=vd.grad)


def errors(got, ref, v, vis, floors=None):
    """Per-row / per-tensor error figures of `got` (out, lse, dq, dk, dv: [B, S, H, hd] / [B, H, S]) against `ref`, and
    the exact-zero violations.  All float64.  floors: {gradient name: norm below which the reference is treated as
    rounding-level} (a gradient that is exactly zero, such as dq when every query sees one key)."""
    floors = floors or {}
    B, S, H, hd = v.shape
    rows = vis.any(-1).expand(B, H, S)                       # [B, H, S]: query has a visible key
    cols = vis.any(-2).expand(B, H, S)                       # key visible to some query
    vabs = v.double().abs().amax(-1).permute(0, 2, 1)        # [B, H, S] max |v| per key
    vmax = torch.where(vis, vabs[:, :, None, :], torch.zeros((), dtype=vabs.dtype, device=vabs.device)).amax(-1)
    e = {}
    oerr = (got["out"].double() - ref["out"]).abs().amax(-1).permute(0, 2, 1)
    e["out"] = float((oerr / vmax.clamp_min(1e-30))[rows].max()) if rows.any() else 0.0
    lse_g, lse_r = got["lse"].double(), ref["lse"]
    e["lse"] = float((lse_g - lse_r)[rows].abs().max()) if rows.any() else 0.0
    e["empty_lse"] = bool((lse_g[~rows] != math.inf).any())
    e["empty_out"] = float(got["out"].double().abs().amax(-1).permute(0, 2, 1)[~rows].max()) if (~rows).any() else 0.0
    for name in ("dq", "dk", "dv"):
        if name in got:
            d = got[name].double() - ref[name]
            e[name] = float(d.norm() / ref[name].norm().clamp_min(floors.get(name, 1e-30)))
    if "dq" in got:
        rn = ref["dq"].norm(dim=-1)                          # [B, S, H]
        floor = (ref["dq"].norm() / math.sqrt(rn.numel())).clamp_min(floors.get("dq", 0.0) / math.sqrt(rn.numel()))
        floor = floor.clamp_min(1e-30)
        e["dq_row"] = float(((got["dq"].double() - ref["dq"]).norm(dim=-1) / torch.maximum(rn, floor)).max())
        e["empty_dq"] = float(got["dq"].double().abs().amax(-1).permute(0, 2, 1)[~rows].max()) if (~rows).any() else 0.0
        e["unseen_dkv"] = float(torch.maximum(got["dk"].double().abs().amax(-1), got["dv"].double().abs().amax(-1))
                                .permute(0, 2, 1)[~cols].max()) if (~cols).any() else 0.0
    return e


def assert_close(got, ref, v, vis, what="", out_tol=OUT_TOL, lse_tol=LSE_TOL, grad_tol=GRAD_TOL, dq_row_tol=DQ_ROW_TOL,
                 floors=None):
    e = errors(got, ref, v, vis, floors)
    print(f"ERR {what} " + " ".join(f"{k}={x:.3g}" if isinstance(x, float) else f"{k}={x}" for k, x in e.items()))
    assert e["out"] <= out_tol, f"{what}: out per-row error {e['out']:.4g} > {out_tol}"
    assert e["lse"] <= lse_tol, f"{what}: lse error {e['lse']:.4g} > {lse_tol}"
    assert not e["empty_lse"], f"{what}: a row with no visible key has a finite lse"
    assert e["empty_out"] == 0.0, f"{what}: a row with no visible key has a non-zero output"
    for name in ("dq", "dk", "dv"):
        if name in e:
            assert e[name] <= grad_tol, f"{what}: {name} relative error {e[name]:.4g} > {grad_tol}"
    if "dq_row" in e:
        assert e["dq_row"] <= dq_row_tol, f"{what}: dq per-row error {e['dq_row']:.4g} > {dq_row_tol}"
        assert e["empty_dq"] == 0.0, f"{what}: a row with no visible key has a non-zero dq"
        assert e["unseen_dkv"] == 0.0, f"{what}: a key no query sees has a non-zero dk / dv"
    return e


# ------------------------------------------------------------------------------------------------
# comparator sensitivity (no GPU)
# ------------------------------------------------------------------------------------------------
def test_comparator_rejects_one_key():
    """The bounds must see one key too many or too few in a row, and an lse that counts one extra zero-score key (the
    weight a padding column of the ragged tail adds)."""
    g = torch.Generator().manual_seed(3)
    B, S, H, hd = 1, 300, 2, 32
    q, k, v, d_o = (torch.randn(B, S, H, hd, generator=g).to(torch.bfloat16) for _ in range(4))
    labels = make_labels("block48", B, S, g)
    vis = visibility(labels, B, S, "cpu")
    ref = reference(q, k, v, vis, hd ** -0.5, d_o)
    same = errors(ref, ref, v, vis)
    assert same["out"] == 0.0 and same["lse"] == 0.0
    i = 100                                               # row of block 2 (keys 0..143 visible)
    extra = vis.clone(); extra[0, 0, i, 144] = True       # first key of the next block
    dropped = vis.clone(); dropped[0, 0, i, 143] = False  # last key of its own block
    for name, mvis in (("extra key", extra), ("dropped key", dropped)):
        bad = reference(q, k, v, mvis, hd ** -0.5, d_o)
        with pytest.raises(AssertionError):
            assert_close(bad, ref, v, vis, what=name)
    bad_lse = dict(ref)
    bad_lse["lse"] = ref["lse"].clone()
    bad_lse["lse"][0, 0, S - 1] = torch.log2(torch.exp2(ref["lse"][0, 0, S - 1]) + 1.0)
    with pytest.raises(AssertionError):
        assert_close(bad_lse, ref, v, vis, what="lse + one key")


# ------------------------------------------------------------------------------------------------
# running the kernels
# ------------------------------------------------------------------------------------------------
def _mask(labels, dev):
    from frankenstein_b200.ops import LabelMask
    if labels is None:
        return None
    return LabelMask(labels[0].to(torch.int32).to(dev), labels[1].to(torch.int32).to(dev))


def _inputs(B, S, H, hd, seed, amp=1.5):
    g = torch.Generator().manual_seed(seed)
    qkv = (torch.randn(B, S, 3 * H * hd, generator=g) * amp).to(torch.bfloat16)
    d_o = torch.randn(B, S, H * hd, generator=g).to(torch.bfloat16)
    return qkv.cuda(), d_o.cuda(), g


def run_ops(qkv, H, labels, d_o, scale=None, rope=None):
    """ops.attention_qkv forward + backward.  Returns (result dict with out / lse / dq / dk / dv as [B, S, H, hd] and
    [B, H, S], the operands the kernels read: q / k after RoPE, v)."""
    from frankenstein_b200 import ops
    B, S, W = qkv.shape
    hd = W // (3 * H)
    x = qkv.clone().requires_grad_(True)
    out = ops.attention_qkv(x * 1.0, H, rope, _mask(labels, qkv.device), scale)
    used, _, lse = out.grad_fn.saved_tensors               # (q and k rotated in place when RoPE is on)
    q, k, v = used.detach().view(B, S, 3, H, hd).clone().unbind(2)
    lse = lse.clone()
    out.backward(d_o)
    dq, dk, dv = x.grad.view(B, S, 3, H, hd).unbind(2)
    got = dict(out=out.detach().view(B, S, H, hd), lse=lse, dq=dq, dk=dk, dv=dv)
    return got, (q, k, v)


def check_case(qkv, H, labels, d_o, what, scale=None, rope=None, rope_ref=None, **tol):
    B, S, W = qkv.shape
    hd = W // (3 * H)
    sc = hd ** -0.5 if scale is None else scale
    got, (q, k, v) = run_ops(qkv, H, labels, d_o, scale, rope)
    vis = visibility(labels, B, S, qkv.device)
    ref = reference(q, k, v, vis, sc, d_o.view(B, S, H, hd))
    if rope_ref is not None:                               # gradients with respect to the unrotated q / k
        ref["dq"], ref["dk"] = rope_ref(ref["dq"]), rope_ref(ref["dk"])
    return got, ref, assert_close(got, ref, v, vis, what, floors=grad_floors(q, k, v, d_o, sc), **tol)


def grad_floors(q, k, v, d_o, scale):
    """1e-3 of each gradient's natural size (|dS| <= |dO| |v| per score): the relative error of a gradient whose
    reference is zero or nearly so (one visible key per query) is measured against that instead."""
    n = d_o.double().norm()
    vm, km, qm = (t.double().norm(dim=-1).max() for t in (v, k, q))
    return dict(dq=1e-3 * scale * n * vm * km, dk=1e-3 * scale * n * vm * qm, dv=1e-3 * n)


gpu = pytest.mark.gpu


@pytest.fixture
def path(request, monkeypatch):
    from frankenstein_b200 import ops
    for name, value in PATHS[request.param].items():
        monkeypatch.setattr(ops, name, value)
    return request.param


# ------------------------------------------------------------------------------------------------
# mask families x shapes x paths
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("path", list(PATHS), indirect=True)
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("S", SHAPES)
def test_masks_hd32(S, kind, path):
    B, H = 2, 2
    qkv, d_o, g = _inputs(B, S, H, 32, 1000 * S + KINDS.index(kind))
    check_case(qkv, H, make_labels(kind, B, S, g), d_o, f"hd32 {path} {kind} S={S}")


@gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("S", SHAPES)
def test_masks_hd64(S, kind):
    B, H = 2, 2
    qkv, d_o, g = _inputs(B, S, H, 64, 1000 * S + KINDS.index(kind) + 7)
    check_case(qkv, H, make_labels(kind, B, S, g), d_o, f"hd64 {kind} S={S}")


@gpu
@pytest.mark.parametrize("hd,path", [(32, "tc"), (32, "tc-staged"), (32, "tc-transposed"), (32, "legacy"), (64, "tc")],
                         indirect=["path"])
@pytest.mark.parametrize("S", [65, 129, 300, 1000])
def test_int32_max_queries_equal_unmasked(S, hd, path):
    """qid = INT32_MAX for every query admits every key: the result must be bit-identical to the unmasked run, and
    right.  (Keys past S in the last tile must not count, whatever the query label.)"""
    B, H = 2, 2
    qkv, d_o, g = _inputs(B, S, H, hd, 77 + S)
    labels = make_labels("int32max", B, S, g)
    got, ref, _ = check_case(qkv, H, labels, d_o, f"int32max hd{hd} {path} S={S}")
    plain, _ = run_ops(qkv, H, None, d_o)
    for name in ("out", "lse", "dq", "dk", "dv"):
        assert torch.equal(got[name], plain[name]), f"{name}: qid = INT32_MAX differs from the unmasked result"


# ------------------------------------------------------------------------------------------------
# many work items per CTA: every sample its own mask, empty items, determinism
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("hd", [32, 64])
def test_many_items_mixed_masks(hd):
    """B = 8, H = 16, S = 640: 384 forward and 640 backward items, above 2 x 148 SMs, so CTAs take several items whose
    tile counts differ a lot, including items with no visible tile (samples 0 and 5 are padding only)."""
    B, H, S = 8, 16, 640
    qkv, d_o, g = _inputs(B, S, H, hd, 640 + hd)
    kinds = ["fullpad", "anticausal", "leftpad", "causal", "random", "fullpad", "independent", "extremes"]
    qid, kid = torch.zeros(B, S, dtype=torch.long), torch.zeros(B, S, dtype=torch.long)
    for b, kind in enumerate(kinds):
        if kind == "fullpad":
            qid[b], kid[b] = -1, I32MAX
        else:
            qq, kk = make_labels(kind, 1, S, g)
            qid[b], kid[b] = qq[0], kk[0]
    got, ref, _ = check_case(qkv, H, (qid, kid), d_o, f"many items hd{hd}")
    for b in (0, 5):
        assert got["out"][b].abs().max().item() == 0.0 and got["dq"][b].abs().max().item() == 0.0
        assert got["dk"][b].abs().max().item() == 0.0 and got["dv"][b].abs().max().item() == 0.0
    again, _ = run_ops(qkv, H, (qid, kid), d_o)
    for name in ("out", "lse", "dq", "dk", "dv"):
        assert torch.equal(got[name], again[name]), f"{name} differs between two identical runs"


# ------------------------------------------------------------------------------------------------
# exact invariants
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("hd,path", [(32, "tc"), (32, "tc-staged"), (32, "tc-transposed"), (32, "legacy"), (64, "tc")],
                         indirect=["path"])
def test_invisible_keys_change_nothing(hd, path):
    """Queries labelled <= 7 cannot see keys labelled > 7: new k / v for those keys leave their out, lse and dq rows
    bit-identical.  Query labels are constant over aligned groups of 32 rows: the forward takes some decisions per warp
    (a row maximum pass, a redone tile), which change the rounding, not the value, of the other rows of the warp."""
    B, S, H = 2, 513, 2
    qkv, d_o, g = _inputs(B, S, H, hd, 91)
    qid = torch.randint(0, 16, (B, (S + 31) // 32), generator=g).repeat_interleave(32, dim=1)[:, :S]
    labels = (qid, torch.randint(0, 16, (B, S), generator=g))
    a, _ = run_ops(qkv, H, labels, d_o)
    pert = qkv.clone().view(B, S, 3, H * hd)
    hidden = (labels[1] > 7).cuda()
    pert[:, :, 1:][hidden] = (torch.randn(int(hidden.sum()), 2, H * hd, generator=g) * 3).to(torch.bfloat16).cuda()
    b_, _ = run_ops(pert.view(B, S, -1), H, labels, d_o)
    sel = (labels[0] <= 7).cuda()                          # [B, S]
    assert sel.any() and hidden.any()
    assert torch.equal(a["out"][sel], b_["out"][sel])
    assert torch.equal(a["dq"][sel], b_["dq"][sel])
    assert torch.equal(a["lse"].permute(0, 2, 1)[sel], b_["lse"].permute(0, 2, 1)[sel])


@gpu
@pytest.mark.parametrize("hd,path", [(32, "tc"), (32, "legacy"), (64, "tc")], indirect=["path"])
@pytest.mark.parametrize("S", [1, 65, 300])
def test_single_key_rows_and_empty_rows_exact(S, hd, path):
    """Row 0 of token causal and row S-1 of anti-causal see one key: out is exactly that key's bf16 v.  Queries
    labelled below every key see nothing: out is exactly zero."""
    B, H = 1, 2
    qkv, d_o, g = _inputs(B, S, H, hd, 5 + S)
    for kind, row in (("causal", 0), ("anticausal", S - 1)):
        got, (q, k, v) = run_ops(qkv, H, make_labels(kind, B, S, g), d_o)
        assert torch.equal(got["out"][:, row], v[:, row]), f"{kind}: row {row} is not its only key's v"
    qid = torch.full((B, S), -5); kid = torch.randint(-4, 9, (B, S), generator=g)
    got, _ = run_ops(qkv, H, (qid, kid), d_o)
    assert got["out"].abs().max().item() == 0.0 and got["dq"].abs().max().item() == 0.0
    assert torch.isinf(got["lse"]).all() and (got["lse"] > 0).all()


# ------------------------------------------------------------------------------------------------
# numerics: scale, large logits, RoPE through the fused inverse rotation
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("hd,path", [(32, "tc"), (32, "tc-staged"), (32, "legacy"), (64, "tc")], indirect=["path"])
@pytest.mark.parametrize("scale", [1.0, 0.05])
def test_scale(scale, hd, path):
    B, S, H = 2, 300, 2
    qkv, d_o, g = _inputs(B, S, H, hd, 13, amp=0.5)
    check_case(qkv, H, make_labels("random", B, S, g), d_o, f"scale {scale} hd{hd} {path}", scale=scale)


@gpu
@pytest.mark.parametrize("hd,path", [(32, "tc"), (32, "tc-staged"), (32, "tc-transposed"), (32, "legacy"), (64, "tc")],
                         indirect=["path"])
def test_large_logits(hd, path):
    """q and k scaled so the scaled scores have a standard deviation of about 30: nearly one-hot rows, the redo path of
    the forward and |lse| of a few hundred in the folded statistics."""
    B, S, H = 2, 513, 2
    amp = math.sqrt(30.0)                                  # std(q.k) * hd^-0.5 = amp^2
    g = torch.Generator().manual_seed(19)
    qk = torch.randn(B, S, 2, H * hd, generator=g) * amp
    vv = torch.randn(B, S, 1, H * hd, generator=g)
    qkv = torch.cat([qk, vv], 2).reshape(B, S, -1).to(torch.bfloat16).cuda()
    d_o = torch.randn(B, S, H * hd, generator=g).to(torch.bfloat16).cuda()
    got, ref, _ = check_case(qkv, H, make_labels("causal", B, S, g), d_o, f"large logits hd{hd} {path}", dq_row_tol=0.2)
    assert ref["lse"][torch.isfinite(ref["lse"])].abs().max() > 100


def _rope_fp64(table, pos, inverse):
    """x [B, S, H, hd] float64 -> rotated by table[pos] (cos, sin per pair), conjugate if inverse."""
    def f(x):
        B, S, H, hd = x.shape
        cs = table.double()[pos]                           # [B, S, hd/2, 2]
        c, s = cs[..., 0][:, :, None], cs[..., 1][:, :, None]
        if inverse:
            s = -s
        xr = x.reshape(B, S, H, hd // 2, 2)
        a, b = xr[..., 0], xr[..., 1]
        return torch.stack([a * c - b * s, a * s + b * c], -1).reshape(B, S, H, hd)
    return f


@gpu
@pytest.mark.parametrize("path", ["tc", "tc-staged", "tc-transposed", "legacy"], indirect=True)
@pytest.mark.parametrize("per_sample", [False, True])
def test_rope_hd32(per_sample, path):
    """RopeSpec at head_dim 32 with an offset (rope[-T:]) and with per-sample positions: q / k rotated by fk_rope, dq / dk
    rotated back inside fk_attn_backward_tc (after the backward on the legacy path)."""
    from frankenstein_b200 import ops
    from frankenstein_b200.brainformer import build_complex_rope_cache
    B, S, H, P = 2, 300, 2, 1024
    qkv, d_o, g = _inputs(B, S, H, 32, 31 + per_sample)
    cache = build_complex_rope_cache(32, P, 10000)
    table = torch.view_as_real(cache).float().contiguous().cuda()
    if per_sample:
        pos = torch.stack([torch.sort(torch.randperm(P, generator=g)[:S])[0] for _ in range(B)]).cuda()
        spec = ops.RopeSpec(table, pos, 0)
    else:
        spec = ops.RopeSpec.from_complex(cache.cuda(), S, last=True)
        pos = (torch.arange(S, device="cuda") + spec.offset).expand(B, S)
    check_case(qkv, H, make_labels("gathered" if per_sample else "block48", B, S, g), d_o, f"rope {per_sample} {path}",
               rope=spec, rope_ref=_rope_fp64(table, pos, inverse=True))


# ------------------------------------------------------------------------------------------------
# the C ABI directly
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("S", [1, 63, 64, 65, 200])
def test_label_ranges_exact(S):
    """fk_attn_label_ranges == per-64-token min / max, ragged tail and int32 extremes included (a tile of INT32_MIN only,
    a tile of INT32_MAX only)."""
    from frankenstein_b200.ops import LabelMask
    g = torch.Generator().manual_seed(S)
    B = 3
    ids = torch.randint(I32MIN, I32MAX, (B, S), generator=g, dtype=torch.int64)
    ids[1] = I32MIN
    ids[2, : min(S, 64)] = I32MAX
    ids[0, -1] = I32MIN
    m = LabelMask(ids.to(torch.int32).cuda())
    nt = (S + 63) // 64
    pad = torch.nn.functional.pad
    lo = -pad(-ids.double(), (0, nt * 64 - S), value=-math.inf).view(B, nt, 64).amax(-1)
    hi = pad(ids.double(), (0, nt * 64 - S), value=-math.inf).view(B, nt, 64).amax(-1)
    assert torch.equal(m.qmin.cpu().long(), lo.long()) and torch.equal(m.qmax.cpu().long(), hi.long())


def _strided(B, S, H, hd, pad_t, pad_b, fill=None, g=None):
    """bf16 [B, S, H, hd] view with token stride H * hd + pad_t and batch stride S * ts + pad_b (pads multiples of 8);
    the gaps hold NaN so that a read outside the view shows."""
    ts = H * hd + pad_t
    bs = S * ts + pad_b
    base = torch.full((B * bs + 64,), float("nan"), dtype=torch.bfloat16)
    x = base.as_strided((B, S, H, hd), (bs, ts, hd, 1))
    if fill is not None:
        x.copy_(fill)
    return base.cuda().as_strided((B, S, H, hd), (bs, ts, hd, 1))


@gpu
@pytest.mark.parametrize("hd,impl", [(32, "tc"), (32, "legacy"), (64, "tc")])
@pytest.mark.parametrize("S", [65, 300])
def test_c_abi_separate_buffers(S, hd, impl):
    """Separate q, k, v, out, dO and gradient tensors, each with its own batch / token stride, through the C entry points
    (forward, fk_attn_aug, backward), against the reference; lse and delta included."""
    from frankenstein_b200 import _lib
    from frankenstein_b200._lib import check, counters, lib, ptr, stream
    B, H = 2, 2
    g = torch.Generator().manual_seed(S + hd)
    vals = [torch.randn(B, S, H, hd, generator=g).to(torch.bfloat16) for _ in range(4)]
    q, k, v, d_o = (_strided(B, S, H, hd, pt, pb, f) for (pt, pb), f in zip(((8, 8), (24, 40), (16, 0), (8, 16)), vals))
    out = _strided(B, S, H, hd, 40, 24)
    dq, dk, dv = (_strided(B, S, H, hd, pt, pb) for pt, pb in ((16, 8), (8, 32), (32, 8)))
    labels = make_labels("extremes", B, S, g)
    m = _mask(labels, "cuda")
    lse = torch.empty(B, H, S, device="cuda")
    delta = torch.empty(B, H, S, device="cuda")
    scale = hd ** -0.5
    margs = (ptr(m.qid), ptr(m.kid), ptr(m.qmin), ptr(m.qmax), ptr(m.kmin), ptr(m.kmax), scale)
    st = lambda t: (t.stride(0), t.stride(1))                                  # noqa: E731
    if impl == "legacy":
        check(lib().fk_attn_forward(ptr(q), ptr(k), ptr(v), ptr(out), ptr(lse), B, H, S, S, hd, *st(q), *st(k), *st(v),
                                    *st(out), *margs, stream()), "fk_attn_forward")
        check(lib().fk_attn_backward(ptr(q), ptr(k), ptr(v), ptr(out), ptr(d_o), ptr(lse), ptr(delta), ptr(dq), ptr(dk),
                                     ptr(dv), B, H, S, S, hd, *st(q), *st(k), *st(v), *st(out), *st(d_o), *st(dq), *st(dk),
                                     *st(dv), *margs, 7, stream()), "fk_attn_backward")
    else:
        check(lib().fk_attn_forward_tc(ptr(q), ptr(k), ptr(v), ptr(out), ptr(lse), B, H, S, hd, *st(q), *st(k), *st(v),
                                       *st(out), *margs, counters(_lib.CTR_ATTN_FWD), stream()), "fk_attn_forward_tc")
        aug = torch.empty(B, H, S, 16, device="cuda", dtype=torch.bfloat16)
        check(lib().fk_attn_aug(ptr(out), ptr(d_o), ptr(lse), ptr(delta), ptr(aug), B, H, S, hd, *st(out), *st(d_o), scale,
                                stream()), "fk_attn_aug")
        for part in (2, 4):
            check(lib().fk_attn_backward_tc(ptr(q), ptr(k), ptr(v), ptr(d_o), 0, 0, 0, (S + 7) // 8 * 8, ptr(lse), ptr(delta),
                                            ptr(aug), ptr(dq), ptr(dk), ptr(dv), B, H, S, hd, *st(q), *st(k), *st(v),
                                            *st(d_o), *st(dq), *st(dk), *st(dv), *margs, 0, 0, 0, 0, part,
                                            counters(_lib.CTR_ATTN_BWD), stream()), "fk_attn_backward_tc")
        check_aug(aug, out, d_o, lse, delta, scale)
    torch.cuda.synchronize()
    vis = visibility(labels, B, S, "cuda")
    ref = reference(q, k, v, vis, scale, d_o)
    got = dict(out=out, lse=lse, dq=dq, dk=dk, dv=dv)
    assert_close(got, ref, v, vis, f"C ABI {impl} hd{hd} S={S}")
    ref_delta = (out.double() * d_o.double()).sum(-1).transpose(1, 2)
    assert (delta.double() - ref_delta).abs().max() <= 1e-5 * (out.double() * d_o.double()).abs().sum(-1).transpose(1, 2).max()


def check_aug(aug, out, d_o, lse, delta, scale):
    """fk_attn_aug: delta = rowsum(dO * O) (fp64 of the same bf16 operands); per row of aug, terms 0-2 sum to
    -lse / (scale log2 e) (-1e30 for an empty row) and terms 3-5 to -delta, to bf16^3 precision; terms 6-15 are zero."""
    a = aug.double()
    ref_delta = (out.double() * d_o.double()).sum(-1).transpose(1, 2)
    mag = (out.double() * d_o.double()).abs().sum(-1).transpose(1, 2)
    assert ((delta.double() - ref_delta).abs() <= 1e-5 * mag + 1e-30).all(), "delta"
    nl = torch.where(torch.isinf(lse), torch.full_like(lse, -1e30), -lse / (scale * LOG2E)).double()
    assert ((a[..., 0:3].sum(-1) - nl).abs() <= 2.0 ** -22 * nl.abs()).all(), "aug lse terms"
    assert ((a[..., 3:6].sum(-1) + delta.double()).abs() <= 2.0 ** -22 * delta.double().abs()).all(), "aug delta terms"
    assert (aug[..., 6:] == 0).all(), "aug padding terms"
