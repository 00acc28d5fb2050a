"""The bandwidth-bound kernels of the training step past their first work unit, through the C ABI.

LayerNorm / add+LayerNorm (layernorm.cu), the QKV/RoPE backward and the stand-alone RoPE (rope.cu), the column sums
and the GELU backward (elementwise.cu) and the patch-embedding backward (gemm_simt.cu) each carry state from one row,
image or k-slice to the next: dgamma / dbeta partials across the rows of a warp, d_cos / d_sin across the images of a
thread, column partials across an unrolled row loop, split-K slices of the weight gradient.  Every shape here is sized
FROM THE DEVICE through a mirror of the launcher's formula, and the test asserts that each warp, thread or split really
handles several units, so a later change to a launch configuration cannot make a test vacuous.

* Reductions are fed data that makes them exact in fp32 in ANY summation order (small integers, powers of two, table
  entries on a grid of 1/4): they are compared BIT FOR BIT with float64 sums.  A lost or doubled row moves such a sum
  by far less than any relative tolerance would notice.
* Per-row outputs are checked element by element against float64 with bounds derived from the operation order, and
  for row invariance: a row computed inside a large M equals, bit for bit, the same row computed alone.
* Every output buffer is pre-filled with NaN; every process-wide option is restored in ``finally``.
"""
import contextlib

import pytest
import torch
import torch.nn.functional as F

from test_kernels_at_scale import _bf16_ulp, _gelu64, _p, _sms, _st
from test_parity_gpu import _set_option, report, tcgen05_must_run
from vit_rpe_rope_b200 import _lib, ops

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BF = torch.bfloat16
F32 = torch.float32
NAN = float("nan")
U = 2.0 ** -24  # unit roundoff of fp32
DT = {F32: _lib.VRR_F32, BF: _lib.VRR_BF16}
ERR_UNSUPPORTED = -2


def _lib_():
    return _lib.load()


def _ints(shape, r, seed, dtype=F32):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(-r, r + 1, shape, generator=g, device=DEV).to(dtype)


def _nan(shape, dtype=F32):
    return torch.full(shape, NAN, device=DEV, dtype=dtype)


def _ceil(a, b):
    return -(-a // b)


def _ratio(err, bound):
    """Worst err / bound (0 where err is 0; NaN, so a failure, where the output was never written)."""
    return torch.where(err == 0, torch.zeros_like(err), err / bound).max().item()


# ===================================================================================== A. LayerNorm

LN_WARPS = 8
LN_E = [100, 192, 256, 384, 512, 768, 1024, 2560]
LN_PAIRS = {"ln": [(F32, F32), (F32, BF), (BF, BF)],          # (x dtype, y dtype)
            "add_ln": [(F32, F32), (BF, BF), (F32, BF)]}      # (branch dtype, y dtype)
EPS = 1e-5


def _ln_bwd_ctas_per_sm(e):
    """Mirror of ln_bwd_ctas_per_sm() in layernorm.cu."""
    n = (200 * 1024) // (2 * LN_WARPS * e * 4 + 1024)
    return max(1, min(6, n))


def _ln_reg_width(e):
    return e in (256, 512, 768, 1024)  # E = 128 NV with the NV the launchers instantiate (2, 4, 6, 8)


def _ln_launch(kind, e, m, reg, minb):
    """(CTAs, warps per CTA) of the launch: mirror of ln_fwd_t, ln_bwd_launch, add_ln_fwd_t and add_ln_bwd_t."""
    sm = _sms()
    if kind.startswith("add_ln") and reg and _ln_reg_width(e):
        if kind == "add_ln_fwd":
            return min(_ceil(m, LN_WARPS), 4 * sm), LN_WARPS
        nv = e // 128
        w, b = (8, 2) if nv <= 4 or minb == 2 else ((8, 1) if minb == 1 or nv > 6 else (12, 1))
        return min(_ceil(m, w), b * sm), w
    if kind.endswith("fwd"):
        return min(_ceil(m, LN_WARPS), 8 * sm), LN_WARPS
    return min(_ceil(m, LN_WARPS), _ln_bwd_ctas_per_sm(e) * sm), LN_WARPS


def _ln_variants(kind, e):
    """(ln_reg, ln_bwd_minb) settings that select different kernels or launch shapes at width e."""
    if kind == "add_ln_bwd" and _ln_reg_width(e):
        return [(0, 3), (1, 1), (1, 2), (1, 3)]
    if kind == "add_ln_fwd" and _ln_reg_width(e):
        return [(0, 3), (1, 3)]
    return [(1, 3)]


def _ln_rows():
    """M giving every warp of every launch variant >= 3 rows: the generic forward (8 SM CTAs x 8 warps) needs the
    most; + 37 leaves a ragged last round."""
    return 3 * 64 * _sms() + 37


def _assert_rows_per_warp(kind, e, m, variants):
    for reg, minb in variants:
        ctas, warps = _ln_launch(kind, e, m, reg, minb)
        assert m // (ctas * warps) >= 3, (kind, e, m, reg, minb, ctas, warps)


@contextlib.contextmanager
def _ln_options(reg, minb):
    try:
        _set_option("ln_reg", reg)
        _set_option("ln_bwd_minb", minb)
        yield
    finally:
        _set_option("ln_reg", 1)
        _set_option("ln_bwd_minb", 3)


def _ln_fwd(kind, x, branch, gamma, beta, ydt):
    m, e = x.shape
    y, mean, rstd = _nan((m, e), ydt), _nan((m,)), _nan((m,))
    if kind == "ln":
        _lib.check(_lib_().vrr_layernorm_fwd(_p(x), _p(gamma), _p(beta), _p(y), _p(mean), _p(rstd), m, e, EPS,
                                             DT[x.dtype], DT[ydt], _st()), "layernorm_fwd")
        return dict(y=y, mean=mean, rstd=rstd)
    x_new = _nan((m, e))
    _lib.check(_lib_().vrr_add_layernorm_fwd(_p(x), _p(branch), _p(x_new), _p(gamma), _p(beta), _p(y), _p(mean),
                                             _p(rstd), m, e, EPS, DT[branch.dtype], DT[ydt], _st()), "add_layernorm_fwd")
    return dict(y=y, mean=mean, rstd=rstd, x_new=x_new)


def _param_grad_bufs(e, adjacent):
    """dgamma / dbeta as the two rows of one [2][E] buffer (the single-memset branch), or as two slices of one
    buffer with a NaN gap between them (certainly not adjacent)."""
    if adjacent:
        buf = _nan((2, e))
        return buf, buf[0], buf[1]
    buf = _nan((2 * e + 32,))
    dg, db = buf[:e], buf[e + 32:]
    assert db.data_ptr() != dg.data_ptr() + 4 * e
    return buf, dg, db


def _ln_bwd(kind, dy, x, gamma, mean, rstd, d_xnew=None, bdt=None, adjacent=True):
    m, e = dy.shape
    buf, dgamma, dbeta = _param_grad_bufs(e, adjacent)
    if kind == "ln":
        dx = _nan((m, e), x.dtype)
        _lib.check(_lib_().vrr_layernorm_bwd(_p(dy), _p(x), _p(gamma), _p(mean), _p(rstd), _p(dx), _p(dgamma),
                                             _p(dbeta), m, e, DT[x.dtype], DT[dy.dtype], _st()), "layernorm_bwd")
        out = dict(dx=dx)
    else:
        dx, d_branch = _nan((m, e)), _nan((m, e), bdt)
        _lib.check(_lib_().vrr_add_layernorm_bwd(_p(dy), _p(d_xnew), _p(x), _p(gamma), _p(mean), _p(rstd), _p(dx),
                                                 _p(d_branch), _p(dgamma), _p(dbeta), m, e, DT[bdt], DT[dy.dtype],
                                                 _st()), "add_layernorm_bwd")
        out = dict(dx=dx, d_branch=d_branch)
    if not adjacent:
        assert torch.isnan(buf[e:e + 32]).all(), "the gap between dgamma and dbeta was written"
    return out, dgamma, dbeta


@pytest.mark.parametrize("e", LN_E)
@pytest.mark.parametrize("kind", ["ln", "add_ln"])
def test_layernorm_param_grads_exact(kind, e):
    """dgamma = sum dy xhat and dbeta = sum dy over M rows, >= 3 rows per warp in every launch variant: integer x, dy
    and mean, rstd = 2^-k (k = 1..3), so xhat and every partial sum are exact and the result equals the float64 sum
    bit for bit in any order - every dtype pair, every (ln_reg, ln_bwd_minb) variant, adjacent and separate
    dgamma / dbeta buffers."""
    m = _ln_rows()
    variants = _ln_variants(kind + "_bwd", e)
    _assert_rows_per_warp(kind + "_bwd", e, m, variants)
    x = _ints((m, e), 8, seed=e)
    mean = _ints((m,), 3, seed=e + 1)
    g = torch.Generator(device=DEV).manual_seed(e + 2)
    rstd = torch.ldexp(torch.ones(m, device=DEV), -torch.randint(1, 4, (m,), generator=g, device=DEV))
    dy = _ints((m, e), 3, seed=e + 3)
    gamma = _ints((e,), 2, seed=e + 4)
    d_xnew = _ints((m, e), 2, seed=e + 5)
    terms = dy.double() * ((x - mean[:, None]) * rstd[:, None]).double()
    assert (terms.abs().sum(0).max().item() * 8) < 2 ** 24  # multiples of 2^-3 below 2^24 * 2^-3: every sum exact
    want_g, want_b = terms.sum(0).float(), dy.double().sum(0).float()
    failures = []
    for xdt, ydt in LN_PAIRS[kind]:
        dyt = dy.to(ydt)
        xt = x.to(xdt) if kind == "ln" else x  # add_ln: x_new is fp32, xdt is the branch dtype
        for reg, minb in variants:
            for adjacent in (True, False):
                with _ln_options(reg, minb):
                    _, dg, db = _ln_bwd(kind, dyt, xt, gamma, mean, rstd, d_xnew=d_xnew, bdt=xdt, adjacent=adjacent)
                for name, got, want in (("dgamma", dg, want_g), ("dbeta", db, want_b)):
                    if not torch.equal(got, want):
                        bad = int((got != want).sum().item())
                        failures.append(f"{xdt}/{ydt} ln_reg {reg} minb {minb} adjacent {adjacent}: {name} "
                                        f"{bad} columns differ")
    assert not failures, "\n".join(failures[:10])


def test_layernorm_width_limit():
    """E = 2560 is the documented maximum; E = 2561 is VRR_ERR_UNSUPPORTED at all four entry points."""
    lib = _lib_()
    m, e = 4, 2561
    x, y, dx, dy = _nan((m, e)), _nan((m, e)), _nan((m, e)), _nan((m, e))
    v, mean, rstd = _nan((e,)), _nan((m,)), _nan((m,))
    pg = _nan((2, e))
    f, b = _lib.VRR_F32, _lib.VRR_F32
    assert lib.vrr_layernorm_fwd(_p(x), _p(v), _p(v), _p(y), _p(mean), _p(rstd), m, e, EPS, f, b, _st()) == ERR_UNSUPPORTED
    assert lib.vrr_layernorm_bwd(_p(dy), _p(x), _p(v), _p(mean), _p(rstd), _p(dx), _p(pg[0]), _p(pg[1]), m, e, f, b,
                                 _st()) == ERR_UNSUPPORTED
    assert lib.vrr_add_layernorm_fwd(_p(x), _p(y), _p(dx), _p(v), _p(v), _p(dy), _p(mean), _p(rstd), m, e, EPS, f, b,
                                     _st()) == ERR_UNSUPPORTED
    assert lib.vrr_add_layernorm_bwd(_p(dy), None, _p(x), _p(v), _p(mean), _p(rstd), _p(dx), _p(y), _p(pg[0]), _p(pg[1]),
                                     m, e, f, b, _st()) == ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert torch.isnan(y).all() and torch.isnan(dx).all() and torch.isnan(pg).all()


def _ln_fwd_bounds(xs, gamma, beta, e, ydt):
    """float64 mean / rstd / y of rows xs (float64, as the kernel reads them) and bounds of the kernel's results.

    mean: a lane sums <= E/32 elements, 5 shuffle levels, the scale by fl(1/E): depth ns = E/32 + 8, so
      |d mean| <= ns u mean|x|.
    var: sum of fl(x - mean')^2 (3u per term) over the same tree, plus n dm^2 from the shifted mean:
      |d var| <= (ns + 6) u var + dm^2 (with the scale and the add of eps);  rstd = rsqrtf(var + eps) (<= 2 ulp = 4u, + u for the add):
      |d rstd| / rstd <= rho = |d var| / (2 (var + eps)) + 5u.
    y = fl(fl(fl(x - mean') rstd') gamma + beta): |d y| <= |gamma| (|xhat| (rho + 3u) + rstd dm (1 + rho))
      + u (|gamma xhat| + |beta|) + u |y|, plus one bf16 ulp for a bf16 output."""
    m64 = xs.mean(1)
    d = xs - m64[:, None]
    var = (d * d).mean(1)
    r64 = (var + EPS) ** -0.5
    ns = _ceil(e, 32) + 8
    dm = ns * U * xs.abs().mean(1)
    rho = ((ns + 6) * U * var + dm * dm) / (2 * (var + EPS)) + 5 * U
    xh = d * r64[:, None]
    g64, b64 = gamma.double(), beta.double()
    y64 = xh * g64 + b64
    by = (g64.abs() * (xh.abs() * (rho + 3 * U)[:, None] + (r64 * dm * (1 + rho))[:, None])
          + U * ((xh * g64).abs() + b64.abs() + y64.abs()))
    if ydt == BF:
        by = by + _bf16_ulp(y64)
    return m64, dm, r64, rho * r64, y64, by


def _ln_bwd_bounds(dy, x, gamma, mean, rstd, d_xnew, e):
    """float64 dx of the LayerNorm backward with the kernel's inputs (stored mean / rstd) and its bound.

    xhat = fl(fl(x - mean) rstd) (2u), gw = fl(dy gamma) (u); c1 = mean(gw), c2 = mean(gw xhat) over the summation
    tree of depth ns = E/32 + 8: |d c1| <= ns u mean|gw|, |d c2| <= (ns + 3) u mean|gw xhat|;
    dx = [r +] rstd (gw - c1 - xhat c2): |d dx| <= rstd (5u S + 2u |xhat c2| + |d c1| + |xhat| |d c2|) + 2u |dx|,
    S = |gw| + |c1| + |xhat c2|; returns the bound of an fp32 output and of a bf16 one (+ one bf16 ulp)."""
    r = rstd.double()[:, None]
    xh = (x.double() - mean.double()[:, None]) * r
    gw = dy.double() * gamma.double()
    c1 = gw.mean(1, keepdim=True)
    c2 = (gw * xh).mean(1, keepdim=True)
    dx = r * (gw - c1 - xh * c2)
    if d_xnew is not None:
        dx = dx + d_xnew.double()
    ns = _ceil(e, 32) + 8
    dc1 = ns * U * gw.abs().mean(1, keepdim=True)
    dc2 = (ns + 3) * U * (gw * xh).abs().mean(1, keepdim=True)
    s = gw.abs() + c1.abs() + (xh * c2).abs()
    b = r * (5 * U * s + 2 * U * (xh * c2).abs() + dc1 + xh.abs() * dc2) + 2 * U * dx.abs()
    return dx, b, b + _bf16_ulp(dx)


def _ln_random_inputs(m, e, seed):
    """Random rows with edge rows: row 1 constant (variance 0, rstd = rsqrt(eps)), row 2 = 1e4 + N(0, 1) (the
    two-pass variance must keep it), row 3 tiny values."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(m, e, generator=g, device=DEV) * 1.5 + 0.25
    x[1] = 0.3
    x[2] = 1e4 + torch.randn(e, generator=g, device=DEV)
    x[3] = x[3] * 1e-3
    branch = torch.randn(m, e, generator=g, device=DEV) * 0.5
    branch[1] = 0.0
    gamma = 1.0 + 0.3 * torch.randn(e, generator=g, device=DEV)
    beta = 0.2 * torch.randn(e, generator=g, device=DEV)
    dy = torch.randn(m, e, generator=g, device=DEV)
    d_xnew = torch.randn(m, e, generator=g, device=DEV) * 0.5
    return x, branch, gamma, beta, dy, d_xnew


def _first_diff(outs_a, outs_b):
    for k in outs_a:
        if not torch.equal(outs_a[k], outs_b[k]):
            return k
    return None


@pytest.mark.parametrize("e", LN_E)
@pytest.mark.parametrize("kind", ["ln", "add_ln"])
def test_layernorm_rows_accuracy_invariance_variants(kind, e):
    """Random data (with a constant row, a 1e4 + N(0, 1) row and a tiny row) at M giving >= 3 rows per warp, every
    dtype pair:
    * y, mean, rstd and dx against float64 element by element within the bounds of the operation order
      (_ln_fwd_bounds, _ln_bwd_bounds);
    * every per-row output (y, mean, rstd, x_new, dx, d_branch) bit-identical across the launch variants (the register
      kernels against the generic ones, ln_bwd_minb 1 / 2 / 3) and to the same rows computed alone (small M);
    * add+LayerNorm backward with and without d_xnew."""
    m = _ln_rows()
    fwd_v, bwd_v = _ln_variants(kind + "_fwd", e), _ln_variants(kind + "_bwd", e)
    _assert_rows_per_warp(kind + "_fwd", e, m, fwd_v)
    _assert_rows_per_warp(kind + "_bwd", e, m, bwd_v)
    x0, branch0, gamma, beta, dy0, d_xnew = _ln_random_inputs(m, e, seed=e)
    rows = torch.tensor([0, 1, 2, 3, 4, m // 2, m - 2, m - 1], device=DEV)
    worst = dict(mean=0.0, rstd=0.0, y=0.0, dx=0.0)
    for xdt, ydt in LN_PAIRS[kind]:
        tag = f"{kind} E={e} {xdt}/{ydt}"
        x = x0.to(xdt) if kind == "ln" else x0
        branch = None if kind == "ln" else branch0.to(xdt)
        fwd = []
        for reg, minb in fwd_v:
            with _ln_options(reg, minb):
                fwd.append(_ln_fwd(kind, x, branch, gamma, beta, ydt))
        ref = fwd[0]
        for (reg, minb), o in zip(fwd_v[1:], fwd[1:]):
            assert _first_diff(ref, o) is None, (tag, "forward variant", reg, minb, _first_diff(ref, o))
        alone = _ln_fwd(kind, x[rows].contiguous(), None if branch is None else branch[rows].contiguous(), gamma, beta,
                        ydt)
        for k, v in alone.items():
            assert torch.equal(v, ref[k][rows]), (tag, "forward row invariance", k)
        xs = ref["x_new"].double() if kind == "add_ln" else x.double()
        if kind == "add_ln":
            assert torch.equal(ref["x_new"], x0 + branch.float())
        m64, dm, r64, drstd, y64, by = _ln_fwd_bounds(xs, gamma, beta, e, ydt)
        em = (ref["mean"].double() - m64).abs()
        er = (ref["rstd"].double() - r64).abs()
        ey = (ref["y"].double() - y64).abs()
        for k, err, bnd in (("mean", em, dm), ("rstd", er, drstd), ("y", ey, by)):
            rt = _ratio(err, bnd)
            worst[k] = max(worst[k], rt)
            assert rt <= 1.0, (tag, k, rt, int((err / bnd).flatten().argmax()))
        # backward with the stored mean / rstd
        dy = dy0.to(ydt)
        xin = ref["x_new"] if kind == "add_ln" else x
        for dxn in ((d_xnew, None) if kind == "add_ln" else (None,)):
            outs = []
            for reg, minb in bwd_v:
                with _ln_options(reg, minb):
                    outs.append(_ln_bwd(kind, dy, xin, gamma, ref["mean"], ref["rstd"], d_xnew=dxn, bdt=xdt)[0])
            for (reg, minb), o in zip(bwd_v[1:], outs[1:]):
                assert _first_diff(outs[0], o) is None, (tag, "backward variant", reg, minb, dxn is None,
                                                         _first_diff(outs[0], o))
            alone = _ln_bwd(kind, dy[rows].contiguous(), xin[rows].contiguous(), gamma, ref["mean"][rows].contiguous(),
                            ref["rstd"][rows].contiguous(), d_xnew=None if dxn is None else dxn[rows].contiguous(),
                            bdt=xdt)[0]
            for k, v in alone.items():
                assert torch.equal(v, outs[0][k][rows]), (tag, "backward row invariance", k, dxn is None)
            dx64, b32, bbf = _ln_bwd_bounds(dy, xin, gamma, ref["mean"], ref["rstd"], dxn, e)
            checks = [("dx", outs[0]["dx"], b32 if outs[0]["dx"].dtype == F32 else bbf)]
            if kind == "add_ln":
                checks.append(("d_branch", outs[0]["d_branch"], b32 if xdt == F32 else bbf))
                assert torch.equal(outs[0]["d_branch"], outs[0]["dx"].to(xdt))
            for k, got, bnd in checks:
                err = (got.double() - dx64).abs()
                rt = _ratio(err, bnd)
                worst["dx"] = max(worst["dx"], rt)
                assert rt <= 1.0, (tag, k, dxn is None, rt, int((err / bnd).flatten().argmax()))
    report(f"layernorm {kind} E={e} M={m}: worst ratio to bound mean {worst['mean']:.3f} rstd {worst['rstd']:.3f} "
           f"y {worst['y']:.3f} dx {worst['dx']:.3f}")


# ===================================================================================== B. RoPE

ROPE_GEOMS = {  # name: (B, N, E, H, dtype)
    "vitb_bf16": (64, 197, 768, 12, BF),
    "vitb_fp32": (64, 197, 768, 12, F32),
    "vitl_bf16": (32, 577, 1024, 16, BF),
    "tiny_fp32": (128, 65, 192, 6, F32),
}
ROPE_MODE = {"none": _lib.ROPE_NONE, "axial": _lib.ROPE_AXIAL, "mixed": _lib.ROPE_MIXED}


def _qkv_rope_bwd_chunk(b, n, e, h, dtype):
    """Mirror of the chunk loop of qkv_rope_bwd() in rope.cu: images per thread (b_chunk)."""
    hd, vec = e // h // 2, 4 if dtype == F32 else 8
    blocks = _ceil(h * n * (hd // vec), 128)
    chunks = 1
    while chunks < b and blocks * chunks < 8 * _sms():
        chunks *= 2
    return _ceil(b, chunks)


def _quarter_table(shape, seed):
    """cos / sin values in {0, +-1/4, +-1/2, +-3/4, +-1} (the kernels do not need cos^2 + sin^2 = 1)."""
    return _ints(shape, 4, seed) * 0.25


def _rope_ref_bwd(dp, pl, cos, sin, mode, b, n, e, h):
    """float64 d_qkv [B*N][3E] and the per-(which, image, head, token) d_cos / d_sin terms [2][B][H][N-1][hd]."""
    dh = e // h
    hd = dh // 2
    c = torch.ones(1, h, n, hd, dtype=torch.float64, device=DEV)
    s = torch.zeros(1, h, n, hd, dtype=torch.float64, device=DEV)
    if mode != "none":
        c[:, :, 1:] = cos.double().view(1, -1, n - 1, hd)
        s[:, :, 1:] = sin.double().view(1, -1, n - 1, hd)
    g1, g2 = dp[:2, ..., :hd].double(), dp[:2, ..., hd:].double()
    dq = torch.cat([g1 * c + g2 * s, g2 * c - g1 * s], -1)
    d_planes = torch.cat([dq, dp[2:].double()], 0)  # [3][B][H][N][Dh]
    d_qkv = d_planes.permute(1, 3, 0, 2, 4).reshape(b * n, 3 * e)
    r1, r2 = pl[:2, ..., :hd].double(), pl[:2, ..., hd:].double()
    x1, x2 = r1 * c + r2 * s, r2 * c - r1 * s
    tc = (g1 * x1 + g2 * x2)[:, :, :, 1:]
    ts = (g2 * x1 - g1 * x2)[:, :, :, 1:]
    return d_qkv, tc, ts


@pytest.mark.parametrize("mode", ["none", "axial", "mixed"])
@pytest.mark.parametrize("geom", list(ROPE_GEOMS))
def test_qkv_rope_bwd_exact(geom, mode):
    """vrr_qkv_rope_bwd with integer planes / d_planes in [-4, 4] and cos / sin on a grid of 1/4: every un-rotated
    value is a multiple of 1/4 below 8 (exact in bf16) and every d_cos / d_sin term a multiple of 1/16, so d_qkv
    (rotated rows, cls rows, v passed through) and d_cos / d_sin (axial: summed over batch and heads, mixed: over the
    batch) match float64 bit for bit.  Each thread walks b_chunk images (asserted from a mirror of the chunk loop);
    d_cos / d_sin adjacent, separate and NULL."""
    b, n, e, h, dtype = ROPE_GEOMS[geom]
    chunk = _qkv_rope_bwd_chunk(b, n, e, h, dtype)
    if geom == "tiny_fp32":
        assert _ceil(b, chunk) >= 64, chunk  # one image per thread, >= 64 image chunks adding into d_cos / d_sin
    else:
        assert chunk >= 4, chunk
    dh, hd = e // h, e // h // 2
    pl = _ints((3, b, h, n, dh), 4, seed=b + n, dtype=dtype)
    dp = _ints((3, b, h, n, dh), 4, seed=b + n + 1, dtype=dtype)
    heads_tab = h if mode == "mixed" else 1
    cos = sin = None
    if mode != "none":
        cos = _quarter_table((heads_tab, n - 1, hd), seed=n + 2)
        sin = _quarter_table((heads_tab, n - 1, hd), seed=n + 3)
    d_qkv64, tc, ts = _rope_ref_bwd(dp, pl, cos, sin, mode, b, n, e, h)
    want_qkv = d_qkv64.to(dtype)
    assert torch.equal(want_qkv.double(), d_qkv64)  # the reference itself is exact in the output type
    if mode != "none":
        dims = (0, 1, 2) if mode == "axial" else (0, 1)
        for t in (tc, ts):
            assert t.abs().sum(dims).max().item() < 2 ** 20  # multiples of 1/16 below 2^24 * 2^-4: every sum exact
        want_c = tc.sum(dims).reshape(heads_tab, n - 1, hd).float()
        want_s = ts.sum(dims).reshape(heads_tab, n - 1, hd).float()
    tab_n = heads_tab * (n - 1) * hd
    layouts = ["none"] if mode == "none" else ["adjacent", "separate", "null"]
    for layout in layouts:
        d_qkv = _nan((b * n, 3 * e), dtype)
        buf = dc = ds = None
        if layout == "adjacent":
            buf = _nan((2 * tab_n,))
            dc, ds = buf[:tab_n], buf[tab_n:]
        elif layout == "separate":
            buf = _nan((2 * tab_n + 64,))
            dc, ds = buf[:tab_n], buf[tab_n + 64:]
        _lib.check(_lib_().vrr_qkv_rope_bwd(_p(dp), _p(pl), _p(cos), _p(sin), _p(d_qkv), _p(dc), _p(ds), b, n, e, h,
                                            ROPE_MODE[mode], DT[dtype], _st()), "qkv_rope_bwd")
        assert torch.equal(d_qkv, want_qkv), (geom, mode, layout, int((d_qkv != want_qkv).sum().item()))
        if dc is not None:
            assert torch.equal(dc.view_as(want_c), want_c), (geom, mode, layout, "d_cos")
            assert torch.equal(ds.view_as(want_s), want_s), (geom, mode, layout, "d_sin")
        if layout == "separate":
            assert torch.isnan(buf[tab_n:tab_n + 64]).all()


def _rope_apply_data(b, h, nr, dh, mode, dtype, seed):
    q = _ints((b, h, nr, dh), 4, seed, dtype)
    k = _ints((b, h, nr, dh), 4, seed + 1, dtype)
    heads_tab = h if mode == "mixed" else 1
    cos = _quarter_table((heads_tab, nr, dh // 2), seed + 2)
    sin = _quarter_table((heads_tab, nr, dh // 2), seed + 3)
    return q, k, cos, sin


@pytest.mark.parametrize("dtype", [BF, F32])
@pytest.mark.parametrize("mode", ["axial", "mixed"])
def test_rope_apply_and_table_grad_exact(mode, dtype):
    """vrr_rope_apply (forward and inverse) with B*H*Nr*Dh/2 >> 2^20 threads, and vrr_rope_table_grad, integer q / k /
    gradients and tables on a grid of 1/4: both exact, compared bit for bit; the table gradient is documented
    deterministic, so two calls are bitwise equal."""
    lib = _lib_()
    b, h, nr, dh = 64, 12, 196, 64
    hd = dh // 2
    assert b * h * nr * hd >= 4 * 2 ** 20
    q, k, cos, sin = _rope_apply_data(b, h, nr, dh, mode, dtype, seed=7 + dh)
    c64 = cos.double().view(1, -1, nr, hd)
    s64 = sin.double().view(1, -1, nr, hd)
    for inverse in (0, 1):
        sg = -s64 if inverse else s64
        qo, ko = _nan(q.shape, dtype), _nan(k.shape, dtype)
        _lib.check(lib.vrr_rope_apply(_p(q), _p(k), _p(cos), _p(sin), _p(qo), _p(ko), b, h, nr, dh, ROPE_MODE[mode],
                                      inverse, DT[dtype], _st()), "rope_apply")
        for got, src in ((qo, q), (ko, k)):
            x1, x2 = src[..., :hd].double(), src[..., hd:].double()
            want = torch.cat([x1 * c64 - x2 * sg, x1 * sg + x2 * c64], -1)
            assert torch.equal(got.double(), want), (mode, dtype, inverse)
    gq = _ints((b, h, nr, dh), 4, seed=11, dtype=dtype)
    gk = _ints((b, h, nr, dh), 4, seed=12, dtype=dtype)
    q1, q2, k1, k2 = q[..., :hd].double(), q[..., hd:].double(), k[..., :hd].double(), k[..., hd:].double()
    a1, a2, b1, b2 = gq[..., :hd].double(), gq[..., hd:].double(), gk[..., :hd].double(), gk[..., hd:].double()
    tc = a1 * q1 + a2 * q2 + b1 * k1 + b2 * k2
    ts = a2 * q1 - a1 * q2 + b2 * k1 - b1 * k2
    dims = (0, 1) if mode == "axial" else (0,)
    for t in (tc, ts):
        assert t.abs().sum(dims).max().item() < 2 ** 24  # integer partial sums below 2^24: exact
    want_c = tc.sum(dims).reshape(cos.shape).float()
    want_s = ts.sum(dims).reshape(sin.shape).float()
    runs = []
    for _ in range(2):
        dc, ds = _nan(cos.shape), _nan(sin.shape)
        _lib.check(lib.vrr_rope_table_grad(_p(q), _p(k), _p(gq), _p(gk), _p(dc), _p(ds), b, h, nr, dh, ROPE_MODE[mode],
                                           DT[dtype], _st()), "rope_table_grad")
        runs.append((dc, ds))
    assert torch.equal(runs[0][0], want_c) and torch.equal(runs[0][1], want_s)
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])


# ===================================================================================== C. column sums and GELU

COLSUM_M = [50432, 36928, 36933]  # multiple of 256; remainder 64 (the tail loop alone in the last block); M % 16 = 5


def _colsum(x, m, c, dtype):
    out = _nan((c,))
    _lib.check(_lib_().vrr_colsum(_p(x), _p(out), m, c, DT[dtype], _st()), "colsum")
    return out


@pytest.mark.parametrize("c", [4, 100, 768, 1000, 3072])
@pytest.mark.parametrize("dtype", [BF, F32])
def test_colsum_exact(dtype, c):
    """vrr_colsum of integers in [-3, 3] (every partial sum an integer below 2^24) equals the float64 sum bit for bit:
    the 8-deep unrolled row loop and its tail, ~200 row blocks of atomics, a ragged last column group (C = 1000) and
    colsum_kernel (C % 8 != 0 in bf16)."""
    for m in COLSUM_M:
        x = _ints((m, c), 3, seed=m + c, dtype=dtype)
        assert torch.equal(_colsum(x, m, c, dtype), x.double().sum(0).float()), (dtype, c, m)


@pytest.mark.parametrize("dtype", [BF, F32])
def test_colsum_misaligned_views_exact(dtype):
    """vrr_colsum on a view at every element offset into a larger buffer (fp32: 4 / 8 / 12 bytes, bf16: 2 .. 8 bytes
    off a 16-byte boundary): the offsets the vector loads cannot take run the element-wise kernel; bit for bit."""
    m, c = 36933, 1000
    esz = 4 if dtype == F32 else 2
    for off in (1, 2, 3) if dtype == F32 else (1, 2, 3, 4):
        buf = torch.zeros(m * c + off, device=DEV, dtype=dtype)
        x = buf[off:].view(m, c)
        x.copy_(_ints((m, c), 3, seed=off, dtype=dtype))
        assert x.data_ptr() % 16 == off * esz
        assert torch.equal(_colsum(x, m, c, dtype), x.double().sum(0).float()), (dtype, off)


@pytest.mark.parametrize("dtype", [BF, F32])
def test_gemm_mul_colsum_misaligned_c_exact(dtype):
    """vrr_gemm_mul_colsum with c a view 4 bytes (fp32) / 2 bytes (bf16) off a 16-byte boundary: the SIMT GEMM, the
    MUL epilogue and the column sums of the stored c, all bit for bit with integer operands."""
    lib = _lib_()
    m, n, k = 1000, 768, 72
    a = _ints((m, k), 1, seed=91, dtype=dtype)
    b = _ints((k, n), 1, seed=92, dtype=dtype)
    mul = _ints((m, n), 2, seed=93, dtype=dtype)
    buf = _nan((m * n + 1,), dtype)
    c = buf[1:].view(m, n)
    assert c.data_ptr() % 16 in (2, 4)
    sums = _nan((n,))
    simt0 = _lib.family_count(_lib.IMPL_SIMT)
    _lib.check(lib.vrr_gemm_mul_colsum(_p(a), _p(b), _p(c), _p(mul), _p(sums), m, n, k, 0, 0, DT[dtype], _st()),
               "mul_colsum")
    assert _lib.family_count(_lib.IMPL_SIMT) > simt0
    want = ((a.double() @ b.double()) * mul.double()).to(dtype)  # |acc| <= 72, |c| <= 144: exact in bf16
    assert torch.equal(c, want)
    assert torch.equal(sums, want.double().sum(0).float())


def _gelu_grad_bound(h):
    """float64 gelu'(h) and the bound of gelu_grad() (elementwise.cu) in fp32, before the output rounding.

    * erf by Abramowitz-Stegun 7.1.26: |d erf| <= 1.5e-7, so Phi is off by <= 0.75e-7;
    * e = __expf(-0.5 h h): <= 2 + floor(1.173 |x|) ulp (x = h^2 / 2), plus the rounding of its argument (u h^2);
    * t = __fdividef(1, fmaf(.)): <= 2 ulp + u; P(t) = poly(t) t (sum i |a_i| <= 16.2, sum |a_i| <= 4.5) carries
      16.2 d t + 5 fma roundings of terms <= 4.5; 1 - erf = P e, so |d (1 - erf)| <= (16.2 eps_t + 23 u) e + P e eps_e + u;
    * gelu' = fmaf(h / sqrt(2 pi), e, Phi): |h| pdf (eps_e + 3u) + d Phi + u |gelu'|."""
    _, dg, cdf, pdf = _gelu64(h)
    h = h.double()
    ah = h.abs()
    e = torch.exp(-0.5 * h * h)
    eps_e = (2 + torch.floor(1.173 * 0.5 * h * h)) * 2.0 ** -23 + U * (h * h + 1)
    eps_t = 2 * 2.0 ** -23 + U
    tail2 = 2 * torch.minimum(cdf, 1 - cdf)  # = P e up to the A-S error
    d_erf = (16.2 * eps_t + 23 * U) * e + (tail2 + 3e-7) * eps_e + U
    d_cdf = 0.5 * d_erf + 0.75e-7 + U
    return dg, ah * pdf * (eps_e + 3 * U) + d_cdf + U * dg.abs() + 2.0 ** -149


@pytest.mark.parametrize("dtype", [BF, F32])
def test_gelu_bwd_vs_float64(dtype):
    """vrr_gelu_bwd at M = 50 000 (ragged last 256-row block), C = 3072: dh against float64 dy gelu'(h) element by
    element (_gelu_grad_bound + the output rounding), db against the float64 sum of the STORED dh within the
    summation-depth bound of the kernel: 32 rows per thread + 8 partials + one atomic per 256-row block."""
    m, c = 50000, 3072
    g = torch.Generator(device=DEV).manual_seed(95)
    h = (torch.randn(m, c, generator=g, device=DEV) * 2.5).to(dtype)
    dy = torch.randn(m, c, generator=g, device=DEV).to(dtype)
    dh, db = _nan((m, c), dtype), _nan((c,))
    _lib.check(_lib_().vrr_gelu_bwd(_p(dy), _p(h), _p(dh), _p(db), m, c, DT[dtype], _st()), "gelu_bwd")
    dg, bdg = _gelu_grad_bound(h.float())
    want = dy.double() * dg
    bound = dy.double().abs() * bdg + (U * want.abs() if dtype == F32 else _bf16_ulp(want))
    err = (dh.double() - want).abs()
    r_dh = _ratio(err, bound)
    depth = 32 + 8 + _ceil(m, 256)
    stored = dh.double()
    err_b = (db.double() - stored.sum(0)).abs()
    b_db = 1.01 * depth * U * stored.abs().sum(0) + 2.0 ** -149
    r_db = _ratio(err_b, b_db)
    report(f"gelu_bwd {dtype} M={m} C={c}: dh worst {r_dh:.3f} of bound, db worst {r_db:.3f} of bound")
    assert r_dh <= 1.0, r_dh
    assert r_db <= 1.0, r_db


def _simt_sweep_values(dtype):
    """fp32: every bf16 value in [-8, 8] (subnormals included: the build does not flush them), 10^6 uniform values in
    [-10, 10] and tails to +-100.  bf16: every bf16 value in [-8, 8] and the tails rounded to bf16."""
    bits = torch.arange(0x0000, 0x4101, dtype=torch.int32)
    pos = bits.to(torch.int16).view(BF).float()
    tails = torch.linspace(8.0, 100.0, 4001)
    v = [pos, -pos[1:], tails, -tails]
    if dtype == F32:
        g = torch.Generator().manual_seed(97)
        v.append(torch.rand(10 ** 6, generator=g) * 20 - 10)
    return torch.cat(v).to(dtype).to(DEV)


@pytest.mark.parametrize("dtype", [F32, BF])
def test_simt_gelu_epilogues_vs_float64(dtype):
    """The SIMT GELU epilogues (fp32 operands, and bf16 under VRR_IMPL_SIMT): BiasEpilogue's gelu (erff) and
    gelu_grad_inplace's gelu' (Abramowitz-Stegun), with acc driven to chosen h (A's first column h, B's first column
    ones: FFMA gives acc = h exactly).  BIAS_GELU: c = h bit for bit, c2 = gelu(h) within erff's 2 ulp, the rounding of
    h / sqrt 2 and of the two products (an absolute term: 1 + erf cancels at negative h, as in the reference formula);
    BIAS_GELU_GRAD: c equal to BIAS_GELU's c2, c2 = gelu'(h) within _gelu_grad_bound and bit-equal to vrr_gelu_bwd with
    dy = 1 (the same device function); BIAS_GELU_ACT: c equal to BIAS_GELU's c2."""
    lib = _lib_()
    hv = _simt_sweep_values(dtype)
    m, n, k = hv.numel(), 8, 8
    a = torch.zeros(m, k, device=DEV, dtype=dtype)
    a[:, 0] = hv
    b = torch.zeros(n, k, device=DEV, dtype=dtype)
    b[:, 0] = 1.0
    bias = torch.zeros(n, device=DEV)
    outs = {}
    prev = _lib.set_impl(_lib.IMPL_SIMT) if dtype == BF else None
    try:
        for epi in (_lib.EPI_BIAS_GELU, _lib.EPI_BIAS_GELU_GRAD, _lib.EPI_BIAS_GELU_ACT):
            c, c2 = _nan((m, n), dtype), _nan((m, n), dtype)
            simt0 = _lib.family_count(_lib.IMPL_SIMT)
            _lib.check(lib.vrr_gemm_ex(_p(a), _p(b), _p(c), _p(c2), _p(bias), m, n, k, 0, 1, DT[dtype], DT[dtype], epi,
                                       0, _st()), f"epilogue {epi}")
            assert _lib.family_count(_lib.IMPL_SIMT) == simt0 + 1
            outs[epi] = (c, c2)
    finally:
        if prev is not None:
            _lib.set_impl(prev)
    h_out, gelu_a = outs[_lib.EPI_BIAS_GELU]
    gelu_b, dgelu = outs[_lib.EPI_BIAS_GELU_GRAD]
    assert torch.equal(h_out, hv[:, None].expand(m, n))
    assert torch.equal(gelu_a, gelu_b) and torch.equal(outs[_lib.EPI_BIAS_GELU_ACT][0], gelu_b)
    ones = torch.ones(m, n, device=DEV, dtype=dtype)
    dh, db = _nan((m, n), dtype), _nan((n,))
    _lib.check(lib.vrr_gelu_bwd(_p(ones), _p(h_out), _p(dh), _p(db), m, n, DT[dtype], _st()), "gelu_bwd")
    assert torch.equal(dh, dgelu)
    g, _, _, _ = _gelu64(hv.float())
    ah = hv.double().abs()
    bg = ah * 2.0 ** -21 + 2 * U * g.abs() + 2.0 ** -149
    dg, bdg = _gelu_grad_bound(hv.float())
    if dtype == BF:
        bg, bdg = bg + _bf16_ulp(g), bdg + _bf16_ulp(dg)
    eg = (gelu_b[:, 0].double() - g).abs()
    edg = (dgelu[:, 0].double() - dg).abs()
    rg, rdg = _ratio(eg, bg), _ratio(edg, bdg)
    report(f"simt gelu sweep {dtype} ({m} values): gelu worst {rg:.3f} of bound, gelu' worst {rdg:.3f} of bound")
    assert rg <= 1.0, ("gelu", hv[int((eg / bg).argmax())].item())
    assert rdg <= 1.0, ("gelu'", hv[int((edg / bdg).argmax())].item())


# ===================================================================================== D. patch-embedding backward

def _patch_splits(b, hw, p, e, c):
    """Mirror of patch_bwd_t (split-K over the B*Np token rows) and launch_gemm's k slice: (splits, kps, empty)."""
    np_ = (hw // p) ** 2
    kd, mtok = c * p * p, b * np_
    tiles = _ceil(e, 64) * _ceil(kd, 64)
    splits = max(1, min(_ceil(2 * _sms(), tiles), mtok // 64))
    kps = _ceil(_ceil(mtok, splits), 16) * 16
    empty = sum(1 for z in range(splits) if z * kps >= mtok)
    return splits, kps, empty


def _patch_ref(img, dtok, p):
    """Exact float64 d_weight [E][C P P], d_bias, d_cls, d_pos [Np][E] of integer data (as fp32)."""
    bsz, np1, e = dtok.shape
    cols = F.unfold(img.double(), p, stride=p).transpose(1, 2).reshape(bsz * (np1 - 1), -1)
    g = dtok[:, 1:].double().reshape(-1, e)
    return ((g.t() @ cols).float(), dtok[:, 1:].double().sum((0, 1)).float(), dtok[:, 0].double().sum(0).float(),
            dtok[:, 1:].double().sum(0).float())


def _patch_bwd_check(bsz, c, hw, p, e, idt, dt, tdt):
    lib = _lib_()
    np_ = (hw // p) ** 2
    img = _ints((bsz, c, hw, hw), 2, seed=hw + c, dtype=idt)
    dtok = _ints((bsz, np_ + 1, e), 2, seed=hw + c + 1, dtype=tdt)
    want_w, want_b, want_cls, want_pos = _patch_ref(img, dtok, p)
    assert want_w.abs().max().item() < 2 ** 24
    for with_w in (True, False):
        for with_pos in (True, False):
            d_w = _nan((e, c * p * p)) if with_w else None
            d_b, d_cls = _nan((e,)), _nan((e,))
            d_pos = _nan((np_, e)) if with_pos else None
            _lib.check(lib.vrr_patch_embed_bwd(_p(img), _p(dtok), _p(d_w), _p(d_b), _p(d_cls), _p(d_pos), bsz, c, hw,
                                               hw, p, e, DT[idt], DT[dt], DT[tdt], _st()), "patch_embed_bwd")
            tag = (bsz, c, hw, p, e, idt, dt, tdt, with_w, with_pos)
            if with_w:
                assert torch.equal(d_w, want_w), (tag, int((d_w != want_w).sum().item()))
            assert torch.equal(d_b, want_b) and torch.equal(d_cls, want_cls), tag
            if with_pos:
                assert torch.equal(d_pos, want_pos), tag


@pytest.mark.parametrize("c", [3, 1])
def test_patch_embed_bwd_fp32_split_k_exact(c):
    """fp32 product path at the ViT-Tiny geometry (B 128, 32 px, P 4, E 192): the FFMA weight gradient split over the
    B*Np token rows with AtomicEpilogue - more than one split, and trailing k-slices that are empty (asserted from a
    mirror of the launch) and must add nothing.  Integer images and d_tokens in [-2, 2]: d_weight, d_bias, d_cls and
    d_pos bit for bit, with and without d_pos and d_weight."""
    bsz, hw, p, e = 128, 32, 4, 192
    splits, kps, empty = _patch_splits(bsz, hw, p, e, c)
    assert splits > 1 and empty > 0, (splits, kps, empty)
    _patch_bwd_check(bsz, c, hw, p, e, F32, F32, F32)


@pytest.mark.parametrize("idt,dt,tdt", [(F32, BF, F32), (BF, BF, F32), (BF, BF, BF)])
def test_patch_embed_bwd_bf16_exact(idt, dt, tdt):
    """The bf16 ABI path with d_weight at the ViT-B geometry (B 64, 224 px, P 16, E 768): the 128 x 128 FFMA tile over
    3 k-splits (asserted), the fp32 images rounded to bf16 in the unfold.  Integer data: bit for bit."""
    bsz, c, hw, p, e = 64, 3, 224, 16, 768
    splits, _, _ = _patch_splits(bsz, hw, p, e, c)
    assert splits > 1, splits
    _patch_bwd_check(bsz, c, hw, p, e, idt, dt, tdt)


@pytest.mark.parametrize("idt", [F32, BF])
def test_patch_unfold_exact(idt):
    """vrr_patch_unfold against torch's unfold of the bf16-rounded images (random, off the bf16 grid), bit for bit."""
    bsz, c, hw, p = 64, 3, 224, 16
    g = torch.Generator(device=DEV).manual_seed(99)
    img = torch.randn(bsz, c, hw, hw, generator=g, device=DEV).to(idt)
    np_, kd = (hw // p) ** 2, c * p * p
    out = _nan((bsz * np_, kd), BF)
    _lib.check(_lib_().vrr_patch_unfold(_p(img), _p(out), bsz, c, hw, hw, p, DT[idt], _st()), "patch_unfold")
    want = F.unfold(img.to(BF).float(), p, stride=p).transpose(1, 2).reshape(bsz * np_, kd).to(BF)
    assert torch.equal(out, want)


def test_patch_embed_fn_backward_vitb_exact():
    """ops.PatchEmbedFn backward at the ViT-B geometry under the autocast dtypes (fp32 images and token stream, bf16
    conv): d_w through the tcgen05 GEMM over the unfolded workspace, d_b, d_cls and d_pos - all exact sums of
    integers, so bit for bit (d_w and d_b rounded once to the bf16 parameter dtype)."""
    bsz, c, hw, p, e = 64, 3, 224, 16, 768
    np_ = (hw // p) ** 2
    img = _ints((bsz, c, hw, hw), 2, seed=101)
    w = _ints((e, c, p, p), 2, seed=102, dtype=BF).requires_grad_(True)
    bias = _ints((e,), 2, seed=103, dtype=BF).requires_grad_(True)
    cls = torch.zeros(1, 1, e, device=DEV, requires_grad=True)
    pos = torch.zeros(1, np_, e, device=DEV, requires_grad=True)
    dtok = _ints((bsz, np_ + 1, e), 2, seed=104)
    with tcgen05_must_run():
        tok = ops.PatchEmbedFn.apply(img, w, bias, cls, pos, p)
        tok.backward(dtok)
    torch.cuda.synchronize()
    want_w, want_b, want_cls, want_pos = _patch_ref(img, dtok, p)
    assert torch.equal(w.grad, want_w.view(e, c, p, p).to(BF))
    assert torch.equal(bias.grad, want_b.to(BF))
    assert torch.equal(cls.grad.view(e), want_cls)
    assert torch.equal(pos.grad.view(np_, e), want_pos)
