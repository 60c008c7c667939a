"""Kernel-level parity of csrc/norm_ops.cu: LayerNorm / RMSNorm forward and backward, the fused residual add + norm, the
partial-sum reduction of dweight / dbias and the SwiGLU gate.

References are computed in float64 on the GPU from exactly the operands the kernels see (bf16 inputs up-cast, fp32 inputs
as they are).  Every comparison is per row (per column for dweight / dbias) and never scaled by the tensor's maximum, so
rows whose scales span six decades each have to be right on their own:
- fp32 outputs: |out - ref| <= rtol * max_row m, m = the magnitude of the terms ref is summed from (|xhat * w| + |b| for
  y; for dx the same with rstd * (|g w| + |mean(g w)| + |xhat * mean(g w xhat)|)), which is what the kernel's rounding
  errors scale with: a row of dx may cancel to well below its terms;
- bf16 outputs: the same plus one bf16 ulp of ref (the kernel rounds its fp32 result once);
- dweight / dbias: |out - ref| <= rtol * sum_r m_rc, m = |g| * (|xhat| + mean(|x|) * rstd) for dweight (see _norm_ref)
  and |g| for dbias: the accumulation bound, which does not depend on how much the sum cancels.
Row counts sit on both sides of the kernels' blocks: 8 rows per forward CTA, and one sweep of the persistent backward
(grid x NORM_BWD_WARPS rows), after which every warp takes a second row and uses the registers it loaded ahead."""
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24        # unit roundoff of fp32
RTOL = 1e-5
NORM_BWD_WARPS = 12     # kNormBwdWarps of csrc/norm_ops.cu: warps per CTA of the persistent norm backward
WIDTHS = [4, 68, 128, 132, 256, 260, 512, 516, 768, 1024]
# (k, off): M = k * S + off, S = one sweep of the backward (fk_norm_backward_grid() * NORM_BWD_WARPS rows)
ROWS = [(0, 1), (0, 7), (0, 9), (1, -1), (1, 0), (1, 1), (3, 5)]
NORM_DTYPES = {          # forward (x -> y) and backward (x, g, dx): g has y's dtype, dx has x's
    "f32-bf16": (torch.float32, torch.bfloat16),
    "f32-f32": (torch.float32, torch.float32),
    "bf16-bf16": (torch.bfloat16, torch.bfloat16),
}


def _rows_id(kv):
    k, off = kv
    return f"M={off}" if k == 0 else f"M={k if k > 1 else ''}S{off:+d}".replace("+0", "")


def _sweep():
    from frankenstein_b200._lib import lib
    return lib().fk_norm_backward_grid() * NORM_BWD_WARPS


def _gen(*key):
    return torch.Generator(device="cuda").manual_seed(zlib.crc32(repr(key).encode()))


def _row_data(M, D, gen, ratio=3.0):
    """rows with scales 10^U(-3, 3) and offsets up to `ratio` times the row's scale"""
    scale = 10.0 ** (torch.rand(M, 1, generator=gen, device="cuda") * 6 - 3)
    offset = (torch.rand(M, 1, generator=gen, device="cuda") * 2 - 1) * ratio * scale
    return torch.randn(M, D, generator=gen, device="cuda") * scale + offset


def _params(D, gen):
    w = 1 + 0.5 * torch.randn(D, generator=gen, device="cuda")
    b = torch.randn(D, generator=gen, device="cuda")
    return w, b


def _f32(v):
    """the fp32 value the kernel receives for a Python float argument"""
    return float(torch.tensor(v, dtype=torch.float32))


class Ref:
    """a float64 reference value and the magnitude of the terms it is summed from (the scale of the kernel's rounding
    errors, which does not shrink where the terms cancel)"""

    def __init__(self, val, mag):
        self.val, self.mag = val, mag

    def __add__(self, other):
        return Ref(self.val + other.val, self.mag + other.mag)


def _norm_ref(x, w, b, eps, rms):
    """float64 y, xhat (Refs) and rstd of LayerNorm (rms=False) / RMSNorm over the last dim of x [M, D].  The kernel's
    error in xhat is absolute, of the order of u * mean(|x|) * rstd (from the fp32 sum behind its mean), not relative
    to |xhat|: an x close to its row's mean has a small xhat with a large relative error.  xhat's magnitude carries that
    term."""
    x = x.double()
    mean = torch.zeros_like(x[:, :1]) if rms else x.mean(-1, keepdim=True)
    rstd = (((x - mean) ** 2).mean(-1, keepdim=True) + _f32(eps)).rsqrt()
    xhat = (x - mean) * rstd
    xw = xhat * w.double()
    bb = b.double() if b is not None else torch.zeros_like(xw[:1])
    return Ref(xw + bb, xw.abs() + bb.abs()), Ref(xhat, xhat.abs() + x.abs().mean(-1, keepdim=True) * rstd), rstd


def _norm_bwd_ref(g, xhat, rstd, w, rms):
    """float64 dx of the norm (a Ref): rstd * (gw - mean(gw) - xhat * mean(gw * xhat)), no mean(gw) term for RMSNorm"""
    xhat = xhat.val
    gw = g.double() * w.double()
    s1 = torch.zeros_like(gw[:, :1]) if rms else gw.mean(-1, keepdim=True)
    s2 = (gw * xhat).mean(-1, keepdim=True)
    return Ref(rstd * (gw - s1 - xhat * s2), rstd * (gw.abs() + s1.abs() + (xhat * s2).abs()))


def _plain(t):
    return Ref(t.double(), t.double().abs())


def _ulp_bf16(v):
    """spacing of bf16 numbers (8 significant bits) at |v|"""
    return torch.exp2(torch.floor(torch.log2(v.abs().clamp_min(2.0 ** -126))) - 7)


def _fail(what, bad, out, ref, tol):
    idx = bad.nonzero()[0].tolist()
    ratio = ((out - ref).abs() / tol).nan_to_num(nan=math.inf)
    return (f"{what}: {int(bad.sum())} of {bad.numel()} out of bounds, first at {idx}: got {out[tuple(idx)].item():.9g}, "
            f"ref {ref[tuple(idx)].item():.9g}, tol {tol.expand_as(out)[tuple(idx)].item():.3g}; worst err/tol "
            f"{ratio.max().item():.3g}")


def check_rows(out, ref, what, rtol=RTOL):
    """|out - ref.val| <= rtol * max_row ref.mag, plus one bf16 ulp of ref.val for a bf16 output"""
    D = ref.val.shape[-1]
    mag = ref.mag.reshape(-1, D)
    ref = ref.val.reshape(-1, D)
    o = out.detach().reshape(-1, D).double()
    tol = rtol * mag.amax(-1, keepdim=True)
    if out.dtype == torch.bfloat16:
        tol = tol + _ulp_bf16(ref)
    bad = ~((o - ref).abs() <= tol)          # NaN counts as out of bounds
    assert not bad.any(), _fail(what, bad, o, ref, tol)


def check_cols(out, ref, mag, what, rtol=RTOL):
    """dweight / dbias: |out - ref| <= rtol * sum_r |term_rc| (the term's magnitude, for dweight |g| * xhat.mag)"""
    o = out.detach().double()
    tol = rtol * mag
    bad = ~((o - ref).abs() <= tol)
    assert not bad.any(), _fail(what, bad, o, ref, tol)


def check_param_grads(dw, db, g, xhat, what=""):
    """dweight = sum_r g * xhat and dbias = sum_r g (db None: no bias)"""
    g = g.double()
    check_cols(dw, (g * xhat.val).sum(0), (g.abs() * xhat.mag).sum(0), f"{what}dw")
    if db is not None:
        check_cols(db, g.sum(0), g.abs().sum(0), f"{what}db")


# ------------------------------------------------------------------------------------------------
# LayerNorm / RMSNorm (ops.layer_norm / ops.rms_norm -> fk_norm_forward, fk_norm_backward, fk_norm_reduce_partials)
# ------------------------------------------------------------------------------------------------
def _grad(t):
    return None if t is None else t.grad


def _run_norm(x, w, b, odt, rms, g):
    from frankenstein_b200 import ops
    eps = 1e-6 if rms else 1e-5
    xd, wd = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    bd = None if b is None else b.clone().requires_grad_(True)
    y = ops.rms_norm(xd, wd, eps, odt) if rms else ops.layer_norm(xd, wd, bd, eps, odt)
    y.backward(g)
    return y, xd, wd, bd, eps


@pytest.mark.parametrize("rms", [False, True], ids=["layer", "rms"])
@pytest.mark.parametrize("dt", list(NORM_DTYPES))
@pytest.mark.parametrize("D", WIDTHS)
@pytest.mark.parametrize("rows", ROWS, ids=_rows_id)
def test_norm(rows, D, dt, rms):
    M = rows[0] * _sweep() + rows[1]
    xdt, odt = NORM_DTYPES[dt]
    gen = _gen("norm", M, D, dt, rms)
    x = _row_data(M, D, gen)
    special = M // 2 if M >= 9 else None
    if special is not None:
        # RMSNorm: an all-zero row; LayerNorm: a constant row whose sum and mean are exact in fp32, so that x - mean = 0
        x[special] = 0.0 if rms else -2.5
    x = x.to(xdt)
    w, b = _params(D, gen)
    b = None if rms else b
    g = torch.randn(M, D, generator=gen, device="cuda").to(odt)
    y, xd, wd, bd, eps = _run_norm(x, w, b, odt, rms, g)
    assert y.dtype == odt and xd.grad.dtype == xdt
    yr, xhat, rstd = _norm_ref(x, w, b, eps, rms)
    check_rows(y, yr, "y")
    check_rows(xd.grad, _norm_bwd_ref(g, xhat, rstd, w, rms), "dx")
    check_param_grads(wd.grad, _grad(bd), g, xhat)
    if special is not None:
        # variance 0: y is the bias exactly (0 for RMSNorm), and dx stays finite
        assert torch.equal(y[special], torch.zeros_like(y[special]) if rms else b.to(odt)), "y of the constant row"
        assert torch.isfinite(xd.grad[special]).all()


@pytest.mark.parametrize("rms", [False, True], ids=["layer", "rms"])
@pytest.mark.parametrize("dt", list(NORM_DTYPES))
def test_norm_many_rows(dt, rms):
    """40000 rows at D = 512: 22-23 rows per warp, dweight / dbias accumulated over all of them"""
    M, D = 40000, 512
    xdt, odt = NORM_DTYPES[dt]
    gen = _gen("norm_many", dt, rms)
    x = _row_data(M, D, gen).to(xdt)
    w, b = _params(D, gen)
    b = None if rms else b
    g = torch.randn(M, D, generator=gen, device="cuda").to(odt)
    y, xd, wd, bd, eps = _run_norm(x, w, b, odt, rms, g)
    yr, xhat, rstd = _norm_ref(x, w, b, eps, rms)
    check_rows(y, yr, "y")
    check_rows(xd.grad, _norm_bwd_ref(g, xhat, rstd, w, rms), "dx")
    check_param_grads(wd.grad, _grad(bd), g, xhat)


@pytest.mark.parametrize("D", [512, 1024])
def test_layer_norm_large_mean(D):
    """rows with |mean| / std = 1e3.  The kernel sums a row in fp32: each lane adds D / 128 float4 groups (D / 32 values)
    in sequence, then five shuffle levels combine the lanes, so the mean carries a relative error of at most
    (D / 32 + 5) * u, u = 2^-24.  x - mean is then exact (Sterbenz), and the error of the mean shifts the whole row's xhat
    by up to (D / 32 + 5) * u * |mean| * rstd = (D / 32 + 5) * u * 1e3.  A row of D >= 512 normal values has max |xhat| > 2,
    so that shift stays below rtol times the row's largest term with rtol = 2 * (D / 32 + 8) * u * 1e3, for y and dx.
    The bound of dweight carries the error of xhat in its terms already (see _norm_ref)."""
    M = _sweep() + 1
    gen = _gen("large_mean", D)
    scale = 10.0 ** (torch.rand(M, 1, generator=gen, device="cuda") * 4 - 2)
    sign = torch.where(torch.rand(M, 1, generator=gen, device="cuda") < 0.5, -1.0, 1.0)
    x = torch.randn(M, D, generator=gen, device="cuda") * scale + sign * 1e3 * scale
    w, b = _params(D, gen)
    g = torch.randn(M, D, generator=gen, device="cuda")
    rtol = 2 * (D / 32 + 8) * U32 * 1e3
    y, xd, wd, bd, eps = _run_norm(x, w, b, torch.float32, False, g)
    yr, xhat, rstd = _norm_ref(x, w, b, eps, False)
    check_rows(y, yr, "y", rtol)
    check_rows(xd.grad, _norm_bwd_ref(g, xhat, rstd, w, False), "dx", rtol)
    check_param_grads(wd.grad, _grad(bd), g, xhat)


@pytest.mark.parametrize("odt", [torch.bfloat16, torch.float32], ids=["bf16", "f32"])
@pytest.mark.parametrize("D", [132, 1024])
def test_layer_norm_without_bias(D, odt):
    M = _sweep() + 1
    gen = _gen("nobias", D, odt)
    x = _row_data(M, D, gen)
    w, _ = _params(D, gen)
    g = torch.randn(M, D, generator=gen, device="cuda").to(odt)
    y, xd, wd, _, eps = _run_norm(x, w, None, odt, False, g)
    yr, xhat, rstd = _norm_ref(x, w, None, eps, False)
    check_rows(y, yr, "y")
    check_rows(xd.grad, _norm_bwd_ref(g, xhat, rstd, w, False), "dx")
    check_param_grads(wd.grad, None, g, xhat)


# ------------------------------------------------------------------------------------------------
# fused residual add + norm (ops.add_layer_norm / ops.add_rms_norm -> fk_add_norm_forward / fk_add_norm_backward)
# ------------------------------------------------------------------------------------------------
def _add_norm(x, delta, w, b, rms, odt):
    from frankenstein_b200 import ops
    eps = 1e-6 if rms else 1e-5
    if rms:
        return ops.add_rms_norm(x, delta, w, eps, odt), eps
    return ops.add_layer_norm(x, delta, w, b, eps, odt), eps


def _add_norm_inputs(M, D, gen, odt, rms):
    x = _row_data(M, D, gen)
    delta = (x.abs().amax(-1, keepdim=True) * torch.randn(M, D, generator=gen, device="cuda")).to(torch.bfloat16)
    w, b = _params(D, gen)
    gy = torch.randn(M, D, generator=gen, device="cuda").to(odt)
    gx = torch.randn(M, D, generator=gen, device="cuda")
    return x, delta, w, None if rms else b, gy, gx


def _leaves(*ts):
    return [None if t is None else t.clone().requires_grad_(True) for t in ts]


@pytest.mark.parametrize("rms", [False, True], ids=["layer", "rms"])
@pytest.mark.parametrize("odt", [torch.bfloat16, torch.float32], ids=["bf16", "f32"])
@pytest.mark.parametrize("D", WIDTHS)
@pytest.mark.parametrize("rows", ROWS, ids=_rows_id)
def test_add_norm(rows, D, odt, rms):
    M = rows[0] * _sweep() + rows[1]
    x, delta, w, b, gy, gx = _add_norm_inputs(M, D, _gen("add_norm", M, D, odt, rms), odt, rms)
    xd, dd, wd, bd = _leaves(x, delta, w, b)
    (xn, y), eps = _add_norm(xd, dd, wd, bd, rms, odt)
    torch.autograd.backward([xn, y], [gx, gy])
    assert xn.dtype == torch.float32 and y.dtype == odt
    assert torch.equal(xn, x + delta.float()), "x_new is not x + float(delta)"
    yr, xhat, rstd = _norm_ref(xn.detach(), w, b, eps, rms)
    check_rows(y, yr, "y")
    check_rows(xd.grad, _norm_bwd_ref(gy, xhat, rstd, w, rms) + _plain(gx), "dx")
    assert dd.grad.dtype == torch.bfloat16 and torch.equal(dd.grad, xd.grad.to(torch.bfloat16)), "d delta is not bf16(dx)"
    check_param_grads(wd.grad, _grad(bd), gy, xhat)


@pytest.mark.parametrize("rms", [False, True], ids=["layer", "rms"])
@pytest.mark.parametrize("D", [68, 512, 1024])
def test_add_norm_broadcast_residual(D, rms):
    """x [1, S, D] broadcast over the batch of delta [B, S, D] (the Encoder's embedding + patch projection): the gradient
    of x is the batch sum of the per-row dx, that of delta the per-row dx itself"""
    B, S = 3, _sweep() // 2 + 3
    gen = _gen("bcast", D, rms)
    x = _row_data(S, D, gen).view(1, S, D)
    delta = (x.abs().amax(-1, keepdim=True) * torch.randn(B, S, D, generator=gen, device="cuda")).to(torch.bfloat16)
    w, b = _params(D, gen)
    b = None if rms else b
    gy = torch.randn(B, S, D, generator=gen, device="cuda").to(torch.bfloat16)
    gx = torch.randn(B, S, D, generator=gen, device="cuda")
    xd, dd, wd, bd = _leaves(x, delta, w, b)
    (xn, y), eps = _add_norm(xd, dd, wd, bd, rms, torch.bfloat16)
    torch.autograd.backward([xn, y], [gx, gy])
    assert tuple(xn.shape) == (B, S, D) and tuple(xd.grad.shape) == (1, S, D)
    assert torch.equal(xn, x + delta.float())
    yr, xhat, rstd = _norm_ref(xn.detach().view(-1, D), w, b, eps, rms)
    check_rows(y, yr, "y")
    dxr = _norm_bwd_ref(gy.view(-1, D), xhat, rstd, w, rms) + _plain(gx.view(-1, D))
    check_rows(dd.grad, dxr, "d delta")
    check_rows(xd.grad, Ref(dxr.val.view(B, S, D).sum(0), dxr.mag.view(B, S, D).sum(0)), "dx (batch sum)")
    check_param_grads(wd.grad, _grad(bd), gy.view(-1, D), xhat)


@pytest.mark.parametrize("D", [260, 768])
def test_add_norm_unused_outputs(D):
    """only y used (the last add+norm of a stack): dx = norm backward alone; only x_new used: dx = g_xnew exactly and
    the parameter gradients are zero"""
    M = _sweep() + 1
    x, delta, w, b, gy, gx = _add_norm_inputs(M, D, _gen("unused", D), torch.bfloat16, False)
    xd, dd, wd, bd = _leaves(x, delta, w, b)
    (xn, y), eps = _add_norm(xd, dd, wd, bd, False, torch.bfloat16)
    y.backward(gy)
    _, xhat, rstd = _norm_ref(xn.detach(), w, b, eps, False)
    check_rows(xd.grad, _norm_bwd_ref(gy, xhat, rstd, w, False), "dx (y only)")
    check_param_grads(wd.grad, _grad(bd), gy, xhat, "y only: ")

    xd, dd, wd, bd = _leaves(x, delta, w, b)
    (xn, y), _ = _add_norm(xd, dd, wd, bd, False, torch.bfloat16)
    xn.backward(gx)
    assert torch.equal(xd.grad, gx) and torch.equal(dd.grad, gx.to(torch.bfloat16))
    assert not wd.grad.any() and not bd.grad.any()


@pytest.mark.parametrize("rms", [False, True], ids=["layer", "rms"])
@pytest.mark.parametrize("D", [132, 1024])
def test_add_norm_backward_without_residual_gradient(D, rms):
    """fk_add_norm_backward with g_res = NULL (x_new has no consumer), through the C entry points: autograd hands the
    wrapper a zero tensor instead, so only a direct call reaches this branch"""
    from frankenstein_b200._lib import check, lib, ptr, stream
    M = 3 * _sweep() + 5
    x, delta, w, b, gy, _ = _add_norm_inputs(M, D, _gen("nores", D, rms), torch.bfloat16, rms)
    eps = 1e-6 if rms else 1e-5
    f32 = dict(device="cuda", dtype=torch.float32)
    xn, mean, rstd = torch.empty(M, D, **f32), torch.empty(M, **f32), torch.empty(M, **f32)
    y = torch.empty(M, D, device="cuda", dtype=torch.bfloat16)
    check(lib().fk_add_norm_forward(ptr(x), ptr(delta), ptr(w), ptr(b), ptr(xn), ptr(y), 1, ptr(mean), ptr(rstd), M, D,
                                    eps, int(rms), 0, stream()), "fk_add_norm_forward")
    nb = lib().fk_norm_backward_grid()
    dx, dx16 = torch.empty(M, D, **f32), torch.empty(M, D, device="cuda", dtype=torch.bfloat16)
    dwp, dbp = torch.empty(nb, D, **f32), (None if rms else torch.empty(nb, D, **f32))
    dw, db = torch.empty(D, **f32), (None if rms else torch.empty(D, **f32))
    check(lib().fk_add_norm_backward(ptr(xn), ptr(gy), 1, None, ptr(w), 0 if rms else ptr(mean), ptr(rstd), ptr(dx),
                                     ptr(dx16), ptr(dwp), ptr(dbp), M, D, int(rms), stream()), "fk_add_norm_backward")
    check(lib().fk_norm_reduce_partials(ptr(dwp), ptr(dbp), nb, D, ptr(dw), ptr(db), stream()), "fk_norm_reduce_partials")
    assert torch.equal(xn, x + delta.float())
    yr, xhat, rstd_r = _norm_ref(xn, w, b, eps, rms)
    check_rows(y, yr, "y")
    check_rows(dx, _norm_bwd_ref(gy, xhat, rstd_r, w, rms), "dx")
    assert torch.equal(dx16, dx.to(torch.bfloat16))
    check_param_grads(dw, db, gy, xhat)


@pytest.mark.parametrize("D", [512, 768])
def test_norm_backward_deterministic(D):
    """two backward passes on the same inputs give bit-identical dx, dweight and dbias (norm and add + norm)"""
    M = 3 * _sweep() + 5
    gen = _gen("determinism", D)
    x, delta, w, b, gy, gx = _add_norm_inputs(M, D, gen, torch.bfloat16, False)
    runs = []
    for _ in range(2):
        _, xd, wd, bd, _ = _run_norm(x, w, b, torch.bfloat16, False, gy)
        xa, dd, wa, ba = _leaves(x, delta, w, b)
        (xn, y), _ = _add_norm(xa, dd, wa, ba, False, torch.bfloat16)
        torch.autograd.backward([xn, y], [gx, gy])
        runs.append([t.grad for t in (xd, wd, bd, xa, dd, wa, ba)])
    for name, a, c in zip(["dx", "dw", "db", "add dx", "add d delta", "add dw", "add db"], *runs):
        assert torch.equal(a, c), name


# ------------------------------------------------------------------------------------------------
# rejections (host side: nothing is launched)
# ------------------------------------------------------------------------------------------------
def test_norm_rejections():
    from frankenstein_b200 import ops
    from frankenstein_b200._lib import FkError, launch_count, lib, ptr, stream
    n0 = launch_count()
    for D in (1028, 66):        # wider than the kernels' 1024 columns; not a multiple of 4
        x = torch.randn(16, D, device="cuda")
        w, b = torch.ones(D, device="cuda"), torch.zeros(D, device="cuda")
        dl = torch.zeros(16, D, device="cuda", dtype=torch.bfloat16)
        for call in (lambda: ops.layer_norm(x, w, b), lambda: ops.rms_norm(x, w),
                     lambda: ops.add_layer_norm(x, dl, w, b), lambda: ops.add_rms_norm(x, dl, w)):
            with pytest.raises(FkError):
                call()
        f = torch.empty(16, device="cuda")
        part = torch.empty(lib().fk_norm_backward_grid(), D, device="cuda")
        assert lib().fk_norm_backward(ptr(x), 0, ptr(x), 0, ptr(w), ptr(f), ptr(f), ptr(x), 0, ptr(part), ptr(part),
                                      16, D, 0, stream()) != 0
        assert lib().fk_add_norm_backward(ptr(x), ptr(x), 0, None, ptr(w), ptr(f), ptr(f), ptr(x), None, ptr(part), None,
                                          16, D, 0, stream()) != 0
    # x_period must divide the row count
    D = 64
    x, w = torch.randn(3, D, device="cuda"), torch.ones(D, device="cuda")
    dl = torch.zeros(10, D, device="cuda", dtype=torch.bfloat16)
    out, f = torch.empty(10, D, device="cuda"), torch.empty(10, device="cuda")
    assert lib().fk_add_norm_forward(ptr(x), ptr(dl), ptr(w), None, ptr(out), ptr(out), 0, ptr(f), ptr(f), 10, D, 1e-5, 0,
                                     3, stream()) != 0
    assert launch_count() == n0


# ------------------------------------------------------------------------------------------------
# SwiGLU gate (fk_swiglu_forward, fk_swiglu_backward, fk_swiglu_backward_blocked)
# ------------------------------------------------------------------------------------------------
SWIGLU_SPECIAL = [0.0, 1e-3, -1e-3, 5.0, -5.0, 20.0, -20.0, 100.0, -100.0]
# For a <= -85, exp(-a) >= e^85 and the kernels' 1 + __expf(-a) exceeds 2^126 from a = -87.3 on, where __fdividef returns
# 0 (and exp(100) is inf): there the kernels flush silu and its derivatives to 0, while the true values are below
# 91 * e^-85 * |g| * |b| < 1.2e-35 * |g| * |b| (|g|, |b| < 15 here).  That band is held to this absolute floor instead.
SWIGLU_FLUSH_A = -85.0
SWIGLU_FLUSH_FLOOR = 1e-32


def _swiglu_inputs(M, H, gen):
    a = torch.randn(M, H, generator=gen, device="cuda") * 3
    flat = a.view(-1)
    i = torch.arange(flat.numel(), device="cuda")
    special = torch.tensor(SWIGLU_SPECIAL, device="cuda")
    flat[i % 3 == 1] = special[(i[i % 3 == 1] // 3) % len(special)]
    band = i % 5 == 2
    flat[band] = -90 + 5 * torch.rand(int(band.sum()), generator=gen, device="cuda")
    b = torch.randn(M, H, generator=gen, device="cuda") * 2
    g = torch.randn(M, H, generator=gen, device="cuda") * 2
    return a.to(torch.bfloat16), b.to(torch.bfloat16), g.to(torch.bfloat16)


def _blocked(h1, h3, block):
    """columns [h1 block 0 | h3 block 0 | h1 block 1 | h3 block 1 | ...], `block` hidden units per block"""
    M, H = h1.shape
    return torch.stack([h1.view(M, H // block, block), h3.view(M, H // block, block)], dim=2).reshape(M, 2 * H)


def _unblocked(h13, block):
    M, H = h13.shape[0], h13.shape[1] // 2
    v = h13.view(M, H // block, 2, block)
    return v[:, :, 0].reshape(M, H), v[:, :, 1].reshape(M, H)


def _check_bf16_ulp(out, ref, slack, what, a):
    """|out - ref| <= one bf16 ulp of ref + slack, and the absolute floor where the kernels flush (a <= -85)"""
    o = out.double()
    tol = _ulp_bf16(ref) + slack
    tol = torch.where(a.double() <= SWIGLU_FLUSH_A, tol.clamp_min(SWIGLU_FLUSH_FLOOR), tol)
    bad = ~((o - ref).abs() <= tol)
    assert not bad.any(), _fail(what, bad, o, ref, tol)


@pytest.mark.parametrize("H", [8, 136, 2048])
@pytest.mark.parametrize("M", [1, 37, 4096])
def test_swiglu(M, H):
    from frankenstein_b200 import gemm, ops
    from frankenstein_b200._lib import check, lib, ptr, stream
    a, b, g = _swiglu_inputs(M, H, _gen("swiglu", M, H))
    hd = torch.cat([a, b], dim=1).requires_grad_(True)
    y = ops.swiglu(hd)
    y.backward(g)

    # forward against the bf16 torch ops it replaces: both round silu(a) to bf16 before the product, and the kernel's
    # approximate exp / division may round it to the neighbouring bf16 value, which moves the product by |b| * ulp(silu)
    s_t = F.silu(a)
    t = s_t * b
    o, tt = y.double(), t.double()
    tol = _ulp_bf16(torch.maximum(o.abs(), tt.abs())) + b.double().abs() * _ulp_bf16(s_t.double())
    tol = torch.where(a.double() <= SWIGLU_FLUSH_A, tol.clamp_min(SWIGLU_FLUSH_FLOOR), tol)
    bad = ~((o - tt).abs() <= tol)
    assert not bad.any(), _fail("swiglu y", bad, o, tt, tol)

    # backward against float64 derivatives of the bf16 inputs; slack: __expf is good to (2 + 1.173 |a|) fp32 ulps,
    # __fdividef to 2, doubled for the products, relative to the terms' magnitudes (1 - sig cancels for a >> 0)
    a64, b64, g64 = a.double(), b.double(), g.double()
    sig = torch.sigmoid(a64)
    rel = (8 + 2.4 * a64.abs()) * 2 * U32
    da = g64 * b64 * sig * (1 + a64 * (1 - sig))
    db = g64 * a64 * sig
    dh1, dh3 = hd.grad[:, :H], hd.grad[:, H:]
    _check_bf16_ulp(dh1, da, rel * (g64 * b64 * sig).abs() * (1 + a64.abs()), "swiglu d h1", a)
    _check_bf16_ulp(dh3, db, rel * db.abs(), "swiglu d h3", a)

    # the blocked layout of the fused w1 | w3 GEMM: the same arithmetic per element, so bit-identical after de-blocking
    w1t = torch.randn(H, 128, device="cuda")
    if H % 128 == 0:
        assert torch.equal(_blocked(w1t.t(), -w1t.t(), 128), gemm._interleave(w1t, -w1t).t())
    for block in sorted({8, 128, H}):
        if H % block:
            continue
        h13 = _blocked(a, b, block)
        dh = torch.full_like(h13, float("nan"))
        check(lib().fk_swiglu_backward_blocked(ptr(h13), ptr(g), ptr(dh), M, H, block, stream()),
              "fk_swiglu_backward_blocked")
        d1, d3 = _unblocked(dh, block)
        assert torch.equal(d1, dh1) and torch.equal(d3, dh3), f"blocked backward, block {block}"


# ------------------------------------------------------------------------------------------------
# model level: an Encoder at dim 768 (norm backward above 512 columns) against the CPU oracle
# ------------------------------------------------------------------------------------------------
def test_encoder_dim768_matches_oracle():
    from frankenstein_b200 import brainformer as bf
    from oracle import brainformer_ref as o
    from tests.test_transformer_gpu import _grads_close, _small_cfg, close
    torch.manual_seed(0)
    cfg = dict(_small_cfg(), dim=768)
    enc = bf.Encoder(bf.MAEConfig(**cfg)).cuda()
    x = torch.randn(3, 64, 16)
    w = torch.randn(3, 128, 768)
    y = enc(x.cuda())
    (y * w.cuda()).sum().backward()
    sd = {k: v.detach().cpu().clone().requires_grad_(v.is_floating_point()) for k, v in enc.state_dict().items()}
    yr = o.encoder_forward(sd, x, cfg)
    (yr * w).sum().backward()
    assert y.dtype == torch.float32 and tuple(y.shape) == (3, 128, 768)
    close(y, yr, what="encoder out")
    _grads_close(enc, sd, ["transformer.emb.weight", "space_embedding", "transformer.h.0.attn.qw.weight",
                           "transformer.h.1.mlp.w2.weight", "transformer.h.0.ln_1.weight", "transformer.h.1.ln_2.bias",
                           "transformer.ln_f.weight", "transformer.ln_f.bias"])
