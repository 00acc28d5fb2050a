"""The persistent tcgen05 kernels past their first work unit, through the C ABI.

``gemm_pair_kernel`` (gemm_tc2.cu) carries a TMA ring, two TMEM accumulator stages, staging-buffer parity and split-K
partial sums from one work unit to the next; ``attn_fwd_ws_kernel`` (attn_fwd_ws.cu) carries double-buffered K/V, a
bias-table row prefetched one item ahead and a polynomial LUT cached across items.  A bug in any of them shows from a
CTA's second unit on, so every shape here is sized FROM THE DEVICE to give each cluster (GEMM: units = m-tiles x
n-tiles x k-splits over SM / 2 clusters) or CTA (attention: B*H items over SM CTAs) several units.

* GEMMs with small-integer operands are exact in fp32 in any summation order (split-K reduce-adds and column-sum
  atomics included), so their outputs are compared BIT FOR BIT with the documented rounding applied on the host.
* Every output buffer is pre-filled with NaN: a tile that is never stored cannot pass.
* Attention is checked per item against float64 torch on the device (same formulas as oracle/attention_np.py, which is
  too slow at these sizes), and for batch invariance: an image computed inside a large batch must equal, bit for bit,
  the same image computed alone (the forward kernels and dQ / dK / dV use no atomics).
"""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import tables_np as T
from test_parity_gpu import report, tcgen05_must_run
from vit_rpe_rope_b200 import _lib, ops

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
BF = torch.bfloat16
NAN = float("nan")
LAYOUTS = [(0, 0), (0, 1), (1, 0), (1, 1)]


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _clusters():
    return _sms() // 2


# ------------------------------------------------------------------------------------- GEMM geometry

def _bn(n):
    return 256 if n > 128 else 128


def _tiles(m, n):
    return -(-m // 256) * -(-n // _bn(n))


def _pick_splits(tiles, num_k, clusters):
    """Mirror of pick_splits() in gemm_tc2.cu (fp32 C only)."""
    if tiles >= 2 * clusters:
        return 1
    best, best_cost = 1, 1e30
    for s in range(1, min(max(num_k // 8, 1), 64) + 1):
        waves = -(-tiles * s // clusters)
        cost = waves * (num_k / s + 6.0)
        if cost < best_cost - 1e-9:
            best, best_cost = s, cost
    return best


def _units(m, n, k, c_f32):
    t = _tiles(m, n)
    return t * (_pick_splits(t, -(-k // 64), _clusters()) if c_f32 else 1)


def _m_for_units(n, factor, ragged=24):
    """An M (multiple of 8, ragged last m-tile) giving >= factor * clusters units at width n without k-splits."""
    tn = -(-n // _bn(n))
    return -(-factor * _clusters() // tn) * 256 - ragged


# ------------------------------------------------------------------------------------- GEMM helpers

def _ints(shape, r, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(-r, r + 1, shape, generator=g, device=DEV).to(BF)


def _operands(m, n, k, ta, tb, r, seed):
    a = _ints((k, m) if ta else (m, k), r, seed)
    b = _ints((n, k) if tb else (k, n), r, seed + 1)
    return a, b


def _exact_acc(a, b, ta, tb):
    """op(A) . op(B) of integer operands in float64 (exact), as fp32 (exact while |acc| < 2^24)."""
    acc = (a.t() if ta else a).double() @ (b.t() if tb else b).double()
    assert acc.abs().max().item() < 2 ** 22
    return acc.float()


def _off_grid_bias(n):
    # k + 1/3 is not a bf16 value: the kernel must round it to bf16 before the add
    return ((torch.arange(n, device=DEV) % 7) - 3).float() + 1.0 / 3.0


def _gemm_ex(a, b, c, m, n, k, ta, tb, c_dtype, epi=_lib.EPI_NONE, c2=None, bias=None, acc=0):
    return _lib.load().vrr_gemm_ex(_p(a), _p(b), _p(c), _p(c2), _p(bias), m, n, k, ta, tb, _lib.VRR_BF16, c_dtype, epi,
                                   acc, _st())


def _mismatch(got, want, n, splits=1):
    """None when bit-identical, else where the first differing element lies (its work unit)."""
    if got.dtype == want.dtype and torch.equal(got, want):
        return None
    bad = ~(got == want)
    cnt = int(bad.sum().item())
    mm, nn = (int(v) for v in bad.nonzero()[0].tolist())
    return (f"{cnt} elements differ; first at (m {mm}, n {nn}) = m-tile {mm // 256}, n-tile {nn // _bn(n)} "
            f"(k-splits {splits}): got {got[mm, nn].item()!r} want {want[mm, nn].item()!r}")


def _c_ref(acc32, c_f32, bias=None, c0=None, mul=None):
    """The kernel's documented rounding of an exact accumulator: bias cast to bf16 first, one rounding to C."""
    x = acc32
    if bias is not None:
        x = x + bias.to(BF).float()
    if mul is not None:
        x = x * mul.float()
    if c_f32:
        return x if c0 is None else (c0.double() + x.double()).float()  # exact: the tests keep |C| < 2^14
    return x.to(BF)


def _run_exact(a, b, m, n, k, ta, tb, c_f32, epi=_lib.EPI_NONE, bias=None, accumulate=False, seed=0):
    """One vrr_gemm_ex call over a NaN-filled (or integer C0) C; returns a mismatch message or None."""
    cdt = torch.float32 if c_f32 else BF
    c0 = _ints((m, n), 3, seed + 7).float() if accumulate else None
    c = c0.clone() if accumulate else torch.full((m, n), NAN, device=DEV, dtype=cdt)
    rc = _gemm_ex(a, b, c, m, n, k, ta, tb, _lib.VRR_F32 if c_f32 else _lib.VRR_BF16, epi, bias=bias,
                  acc=1 if accumulate else 0)
    if rc != 0:
        return f"rc {rc}: {_lib.last_error()}"
    want = _c_ref(_exact_acc(a, b, ta, tb), c_f32, bias if epi == _lib.EPI_BIAS else None, c0)
    splits = _pick_splits(_tiles(m, n), -(-k // 64), _clusters()) if c_f32 else 1
    return _mismatch(c, want, n, splits)


# ------------------------------------------------------------------------------------- A1: ragged and switch sizes

@pytest.mark.parametrize("c_f32", [0, 1])
@pytest.mark.parametrize("ta,tb", LAYOUTS)
def test_gemm_integer_exact_ragged_shapes(ta, tb, c_f32):
    """Every layout x C type at ragged M, the BN 128 -> 256 switch (N 128 / 136), and K from one k-block to 65: plain,
    BIAS (off-grid fp32 bias) and, for fp32 C, accumulate over an integer C0.  Bit-exact."""
    ms = [8, 248, 264, 384] if ta else [1, 8, 255, 257, 383]  # trans_a stores A [K][M]: M % 8 == 0
    ns = [8, 128, 136, 264] + ([4, 36] if c_f32 and tb else [])
    failures = []
    with tcgen05_must_run():
        for m in ms:
            for n in ns:
                for k in (8, 72, 520, 4104):
                    a, b = _operands(m, n, k, ta, tb, 1 if k > 1000 else 3, seed=m * 7 + n * 3 + k)
                    cases = [("plain", _lib.EPI_NONE, None, False)]
                    if n % 8 == 0:
                        cases.append(("bias", _lib.EPI_BIAS, _off_grid_bias(n), False))
                    if c_f32:
                        cases.append(("accumulate", _lib.EPI_NONE, None, True))
                        if n % 8 == 0:
                            cases.append(("bias+accumulate", _lib.EPI_BIAS, _off_grid_bias(n), True))
                    for what, epi, bias, accum in cases:
                        msg = _run_exact(a, b, m, n, k, ta, tb, c_f32, epi, bias, accum, seed=k)
                        if msg:
                            failures.append(f"M {m} N {n} K {k} {what}: {msg}")
    assert not failures, "\n".join(failures[:10])


# ------------------------------------------------------------------------------------- A2: many units per cluster

@pytest.mark.parametrize("n,k", [(3072, 768), (768, 3072)])  # ViT-B fc1 and fc1's dX
@pytest.mark.parametrize("ta,tb", LAYOUTS)
def test_gemm_integer_exact_many_units(ta, tb, n, k):
    """>= 4 units per cluster (both accumulator stages reused, acc_phase wrapping, staging parity over many chunks),
    bf16 C, plain and BIAS: the whole output bit for bit."""
    m = _m_for_units(n, 4)
    assert _units(m, n, k, False) >= 4 * _clusters()
    a, b = _operands(m, n, k, ta, tb, 3, seed=n + k)
    with tcgen05_must_run():
        msgs = [_run_exact(a, b, m, n, k, ta, tb, 0),
                _run_exact(a, b, m, n, k, ta, tb, 0, _lib.EPI_BIAS, _off_grid_bias(n))]
    assert msgs == [None, None], msgs


# ------------------------------------------------------------------------------------- A3: fp32 C split-K regimes

def _regime_shape(regime):
    cl = _clusters()
    if regime == "no_split":  # tiles >= 2 clusters: one split, plain TMA store
        return _m_for_units(2048, 2), 2048, 1024
    if regime == "split_one_wave":  # tiles < clusters, large K: the weight-gradient shapes
        return 3072, 768, 6304
    # clusters < tiles < 2 clusters with large K: split AND several units per cluster
    return -(-int(1.4 * cl) // 10) * 256, 2560, 4096


@pytest.mark.parametrize("ta,tb", [(1, 0), (0, 1)])
@pytest.mark.parametrize("regime", ["no_split", "split_one_wave", "split_multi_wave"])
def test_gemm_fp32_split_k_regimes_exact(regime, ta, tb):
    """fp32 C (weight gradients): split-K partial sums combined by TMA reduce-add after a memset, gradient
    accumulation (accumulate = 1) over an integer C0, and the bias joining exactly one k-split.  Integer operands keep
    every partial sum exact, so the result is bit-exact in any reduction order."""
    m, n, k = _regime_shape(regime)
    cl = _clusters()
    tiles = _tiles(m, n)
    splits = _pick_splits(tiles, -(-k // 64), cl)
    if regime == "no_split":
        assert tiles >= 2 * cl and splits == 1
    elif regime == "split_one_wave":
        assert tiles < cl and splits > 1 and tiles * splits <= cl, (tiles, splits)
    else:
        assert cl < tiles < 2 * cl and splits > 1 and tiles * splits > cl, (tiles, splits)
    r = 3 if 9 * k < 2 ** 13 else 1  # |acc| < 2^13: acc + bf16(bias) (9 fraction bits) stays exact in fp32
    a, b = _operands(m, n, k, ta, tb, r, seed=m + k)
    bias = _off_grid_bias(n)
    with tcgen05_must_run():
        msgs = {what: _run_exact(a, b, m, n, k, ta, tb, 1, epi, bs, acc)
                for what, epi, bs, acc in (("plain", _lib.EPI_NONE, None, False), ("accumulate", _lib.EPI_NONE, None, True),
                                           ("bias", _lib.EPI_BIAS, bias, False), ("bias+accumulate", _lib.EPI_BIAS, bias, True))}
    assert all(v is None for v in msgs.values()), msgs


# ------------------------------------------------------------------------------------- A4: every epilogue

def _gelu64(h):
    h = h.double()
    phi_c = 0.5 * (1.0 + torch.special.erf(h / math.sqrt(2.0)))
    pdf = torch.exp(-0.5 * h * h) / math.sqrt(2.0 * math.pi)
    return h * phi_c, phi_c + h * pdf, phi_c, pdf


def _bf16_ulp(y):
    y = y.double().abs()
    _, e = torch.frexp(torch.where(y > 0, y, torch.full_like(y, 2.0 ** -126)).clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(y), (e - 8).to(torch.int64))


def _gelu_bounds(h):
    """Error bounds of gelu_and_grad2 (gemm_tc2.cu): one bf16 ulp of the result (the output rounding, plus any fp32
    error below half an ulp), the Abramowitz-Stegun 7.1.26 error |d erfc| <= 1.5e-7 (Phi off by <= 0.75e-7, gelu by
    <= 0.75e-7 |h|), and the fp32 evaluation of the tail erfc/2 = poly(t) t exp(-h^2/2) with rcp.approx / ex2.approx
    (<= 2^-21 relative) and of the products (2^-23)."""
    g, dg, cdf, pdf = _gelu64(h)
    ah = h.double().abs()
    tail = torch.minimum(cdf, 1.0 - cdf)
    bg = _bf16_ulp(g) + ah * (0.75e-7 + 2.0 ** -21 * tail + 2.0 ** -23)
    bdg = _bf16_ulp(dg) + 0.75e-7 + 2.0 ** -21 * (tail + ah * pdf) + 2.0 ** -23
    return g, dg, bg, bdg


def _sweep_values():
    """Every normal bf16 value in [-8, 8], zero, and a few outside.  Subnormal bf16 inputs are left out: the tensor
    cores flush them, so acc (= h) would not be h."""
    bits = torch.arange(0x0080, 0x4101, dtype=torch.int32)  # 2^-126 .. 8.0
    pos = bits.to(torch.int16).view(BF)
    extra = torch.tensor([9.0, 10.0, 12.0, 16.0, 30.0, 100.0], dtype=BF)
    v = torch.cat([torch.zeros(1, dtype=BF), pos, -pos, extra, -extra])
    return v.to(DEV)


def test_gelu_epilogue_sweep_vs_float64():
    """BIAS_GELU and BIAS_GELU_GRAD with acc driven to chosen values: A's first column holds h, B's first column is
    ones, everything else zero, bias 0.  h comes back bit for bit; gelu(h) and gelu'(h) within the bounds of the
    method (_gelu_bounds), element by element; and the three GELU epilogues agree bit for bit."""
    hv = _sweep_values()
    m, n, k = hv.numel(), 8, 8
    a = torch.zeros(m, k, device=DEV, dtype=BF)
    a[:, 0] = hv
    b = torch.zeros(n, k, device=DEV, dtype=BF)
    b[:, 0] = 1.0
    bias = torch.zeros(n, device=DEV)
    outs = {}
    with tcgen05_must_run():
        for epi in (_lib.EPI_BIAS_GELU, _lib.EPI_BIAS_GELU_GRAD, _lib.EPI_BIAS_GELU_ACT):
            c = torch.full((m, n), NAN, device=DEV, dtype=BF)
            c2 = torch.full((m, n), NAN, device=DEV, dtype=BF)
            _lib.check(_gemm_ex(a, b, c, m, n, k, 0, 1, _lib.VRR_BF16, epi, c2=c2, bias=bias), f"epilogue {epi}")
            outs[epi] = (c, c2)
    h_out, gelu_a = outs[_lib.EPI_BIAS_GELU]
    gelu_b, dgelu = outs[_lib.EPI_BIAS_GELU_GRAD]
    assert torch.equal(h_out, hv[:, None].expand(m, n))
    assert torch.equal(gelu_a, gelu_b) and torch.equal(outs[_lib.EPI_BIAS_GELU_ACT][0], gelu_b)
    g, dg, bg, bdg = _gelu_bounds(hv.float())
    eg = (gelu_b[:, 0].double() - g).abs()
    edg = (dgelu[:, 0].double() - dg).abs()
    normal = lambda y: y.abs() >= 2.0 ** -126  # noqa: E731  (ulps of a result that underflows mean nothing)
    ulps_g = (eg / _bf16_ulp(g))[normal(g)].max().item()
    ulps_dg = (edg / _bf16_ulp(dg))[normal(dg)].max().item()
    rg, rdg = (eg / bg).max().item(), (edg / bdg).max().item()
    report(f"gelu sweep ({m} values): gelu worst {ulps_g:.2f} ulp ({rg:.2f} of bound), gelu' worst {ulps_dg:.2f} ulp "
           f"({rdg:.2f} of bound)")
    worst = int((eg / bg).argmax())
    assert rg <= 1.0, ("gelu", hv[worst].item(), gelu_b[worst, 0].item(), g[worst].item())
    worst = int((edg / bdg).argmax())
    assert rdg <= 1.0, ("gelu'", hv[worst].item(), dgelu[worst, 0].item(), dg[worst].item())


@pytest.mark.parametrize("shape", ["ragged", "many_units"])
def test_gemm_epilogues_exact_and_consistent(shape):
    """BIAS (bf16 C), BIAS_GELU, BIAS_GELU_GRAD, BIAS_GELU_ACT and MUL with integer operands: h bit for bit where it is
    an output, MUL bit for bit, gelu(h) bitwise identical across the three GELU epilogues and within the method's
    bound of float64, gelu'(h) within its bound."""
    m, n, k = (383, 136, 520) if shape == "ragged" else (_m_for_units(3072, 4), 3072, 768)
    a, b = _operands(m, n, k, 0, 1, 1, seed=17)  # |acc| ~ 20 typical: h spans GELU's curved range and both tails
    bias = _off_grid_bias(n) * 0.25
    acc = _exact_acc(a, b, 0, 1)
    h = (acc + bias.to(BF).float()).to(BF)
    res = {}
    with tcgen05_must_run():
        for epi in (_lib.EPI_BIAS, _lib.EPI_BIAS_GELU, _lib.EPI_BIAS_GELU_GRAD, _lib.EPI_BIAS_GELU_ACT):
            c = torch.full((m, n), NAN, device=DEV, dtype=BF)
            c2 = torch.full((m, n), NAN, device=DEV, dtype=BF)
            _lib.check(_gemm_ex(a, b, c, m, n, k, 0, 1, _lib.VRR_BF16, epi, c2=c2, bias=bias), f"epilogue {epi}")
            res[epi] = (c, c2)
        mul = _ints((m, n), 3, seed=19)
        cm = torch.full((m, n), NAN, device=DEV, dtype=BF)
        _lib.check(_gemm_ex(a, b, cm, m, n, k, 0, 1, _lib.VRR_BF16, _lib.EPI_MUL, c2=mul), "MUL")
    assert _mismatch(res[_lib.EPI_BIAS][0], h, n) is None
    assert _mismatch(res[_lib.EPI_BIAS_GELU][0], h, n) is None
    assert _mismatch(cm, (acc * mul.float()).to(BF), n) is None
    gl = res[_lib.EPI_BIAS_GELU_GRAD][0]
    assert torch.equal(res[_lib.EPI_BIAS_GELU][1], gl) and torch.equal(res[_lib.EPI_BIAS_GELU_ACT][0], gl)
    g, dg, bg, bdg = _gelu_bounds(h.float())
    assert ((gl.double() - g).abs() <= bg).all()
    assert ((res[_lib.EPI_BIAS_GELU_GRAD][1].double() - dg).abs() <= bdg).all()


@pytest.mark.parametrize("m", [257, 383, "many_units"])
def test_gemm_mul_colsum_exact(m):
    """vrr_gemm_mul_colsum with every stored value a bf16 integer below 256: the stored tile and the column sums
    (fp32 atomics of integers < 2^24) are exact in any order and must match bit for bit; rows past M add nothing."""
    n, k = 768, 72
    if m == "many_units":
        m = _m_for_units(n, 4)
        assert _units(m, n, k, False) >= 4 * _clusters()
    a, b = _operands(m, n, k, 0, 0, 1, seed=m)  # |acc| <= 72, |acc * mul| <= 216
    mul = _ints((m, n), 3, seed=m + 1)
    c = torch.full((m, n), NAN, device=DEV, dtype=BF)
    sums = torch.full((n,), NAN, device=DEV)
    with tcgen05_must_run():
        _lib.check(_lib.load().vrr_gemm_mul_colsum(_p(a), _p(b), _p(c), _p(mul), _p(sums), m, n, k, 0, 0, 1, _st()),
                   "mul_colsum")
    want = (_exact_acc(a, b, 0, 0) * mul.float()).to(BF)
    assert _mismatch(c, want, n) is None
    assert torch.equal(sums, want.double().sum(0).float())


# ------------------------------------------------------------------------------------- A6: random data

# Worst c observed on a B200 (four layouts, M 6376 N 3072 K 768): 1.83e-3 - the fp32 accumulation error stays far
# below the worst case K 2^-24 |A||B|; the bar keeps 4x headroom over that.
C_RANDOM = 8e-3


@pytest.mark.parametrize("ta,tb", LAYOUTS)
def test_gemm_random_data_vs_float64(ta, tb):
    """Non-integer data at a multi-unit shape, element by element against float64:
    |got - ref| <= 2^-8 |ref| + C_RANDOM * K * 2^-24 * (|A| . |B|) - the bf16 output rounding plus the worst-case fp32
    accumulation error scaled by C_RANDOM."""
    n, k = 3072, 768
    m = _m_for_units(n, 4)
    g = torch.Generator(device=DEV).manual_seed(23 + 2 * ta + tb)
    a = torch.randn((k, m) if ta else (m, k), generator=g, device=DEV).to(BF)
    b = torch.randn((n, k) if tb else (k, n), generator=g, device=DEV).to(BF)
    c = torch.full((m, n), NAN, device=DEV, dtype=BF)
    with tcgen05_must_run():
        _lib.check(_gemm_ex(a, b, c, m, n, k, ta, tb, _lib.VRR_BF16), "gemm")
    oa, ob = (a.t() if ta else a).double(), (b.t() if tb else b).double()
    ref = oa @ ob
    mag = oa.abs() @ ob.abs()
    err = (c.double() - ref).abs()
    need = ((err - 2.0 ** -8 * ref.abs()).clamp_min(0) / (k * 2.0 ** -24 * mag)).max().item()
    report(f"gemm random ta={ta} tb={tb} M={m} N={n} K={k}: worst accumulation-error ratio c = {need:.3e}")
    assert need <= C_RANDOM, need


# ------------------------------------------------------------------------------------- E: misaligned operands

def test_gemm_misaligned_operand_runs_simt():
    """A bf16 operand that is a contiguous view at an 8-byte offset cannot feed TMA: under VRR_IMPL_AUTO the call runs
    the SIMT kernel (correct result, SIMT counter advances), under VRR_IMPL_TCGEN05 it is VRR_ERR_UNSUPPORTED."""
    lib = _lib.load()
    m, n, k = 96, 64, 72
    buf = torch.zeros(m * k + 4, device=DEV, dtype=BF)
    a = buf[4:].view(m, k)
    a.copy_(_ints((m, k), 1, seed=31))  # |acc| <= 72, |acc * mul| <= 144: every value exact in bf16
    assert a.data_ptr() % 16 == 8
    b = _ints((n, k), 1, seed=32)
    acc = _exact_acc(a, b, 0, 1)
    want = acc.to(BF)
    for epi in (_lib.EPI_NONE, _lib.EPI_BIAS):
        bias = _off_grid_bias(n) if epi == _lib.EPI_BIAS else None
        c = torch.full((m, n), NAN, device=DEV, dtype=BF)
        simt0 = _lib.family_count(_lib.IMPL_SIMT)
        _lib.check(_gemm_ex(a, b, c, m, n, k, 0, 1, _lib.VRR_BF16, epi, bias=bias), "misaligned gemm")
        assert _lib.family_count(_lib.IMPL_SIMT) == simt0 + 1
        assert torch.equal(c, want if bias is None else (acc + bias.to(BF).float()).to(BF))
    simt0 = _lib.family_count(_lib.IMPL_SIMT)
    assert torch.equal(ops._gemm(a, b, False, True, BF), want)
    assert _lib.family_count(_lib.IMPL_SIMT) == simt0 + 1
    mul = _ints((m, n), 2, seed=33)
    c = torch.full((m, n), NAN, device=DEV, dtype=BF)
    sums = torch.full((n,), NAN, device=DEV)
    _lib.check(lib.vrr_gemm_mul_colsum(_p(a), _p(b), _p(c), _p(mul), _p(sums), m, n, k, 0, 1, 1, _st()), "mul_colsum")
    want_m = (want.float() * mul.float()).to(BF)
    assert torch.equal(c, want_m) and torch.equal(sums, want_m.double().sum(0).float())
    prev = _lib.set_impl(_lib.IMPL_TCGEN05)
    try:
        c = torch.full((m, n), NAN, device=DEV, dtype=BF)
        assert _gemm_ex(a, b, c, m, n, k, 0, 1, _lib.VRR_BF16) == -2  # VRR_ERR_UNSUPPORTED
    finally:
        _lib.set_impl(prev)


# ------------------------------------------------------------------------------------- B: direct-store epilogues

@pytest.mark.parametrize("rope", ["none", "axial", "mixed"])
@pytest.mark.parametrize("b,n,e,h", [(32, 197, 768, 12), (8, 577, 1024, 16)])
def test_qkv_rope_integer_many_units(b, n, e, h, rope):
    """QkvRopeEpi2 over many units (warp tiles that cross an image boundary take the per-row store): integer x and w,
    NaN-filled planes.  No RoPE: bit for bit.  RoPE: within one bf16 ulp of the float64 rotation of the exact
    accumulator, plus the fp32 evaluation of x1 c - x2 s (two products and a sum: 2^-22 (|x1 c| + |x2 s|))."""
    assert _tiles(b * n, 3 * e) >= 2 * _clusters()
    x = _ints((b * n, e), 3, seed=41)
    w = _ints((3 * e, e), 3, seed=42)
    cos = sin = None
    mode = {"none": _lib.ROPE_NONE, "axial": _lib.ROPE_AXIAL, "mixed": _lib.ROPE_MIXED}[rope]
    if rope != "none":
        g = torch.Generator(device=DEV).manual_seed(43)
        ang = torch.rand(*((n - 1, 32) if rope == "axial" else (h, n - 1, 32)), generator=g, device=DEV) * 6.0
        cos, sin = torch.cos(ang), torch.sin(ang)
    planes = torch.full((3, b, h, n, 64), NAN, device=DEV, dtype=BF)
    with tcgen05_must_run():
        _lib.check(_lib.load().vrr_qkv_rope_fwd(_p(x), _p(w), _p(cos), _p(sin), _p(planes), b, n, e, h, mode, 1, _st()),
                   "qkv_rope_fwd")
    acc = (x.double() @ w.double().t()).view(b, n, 3, h, 64).permute(2, 0, 3, 1, 4)  # exact
    if rope == "none":
        assert torch.equal(planes, acc.float().to(BF))
        return
    c64 = cos.double().view(1, 1, n - 1, 32) if rope == "axial" else cos.double().view(1, h, n - 1, 32)
    s64 = sin.double().view(1, 1, n - 1, 32) if rope == "axial" else sin.double().view(1, h, n - 1, 32)
    want = acc.clone()
    fp32_err = torch.zeros_like(acc)
    for which in (0, 1):
        x1, x2 = acc[which, :, :, 1:, :32], acc[which, :, :, 1:, 32:]
        want[which, :, :, 1:, :32] = x1 * c64 - x2 * s64
        want[which, :, :, 1:, 32:] = x1 * s64 + x2 * c64
        mag = x1.abs() * c64.abs() + x2.abs() * s64.abs()
        fp32_err[which, :, :, 1:, :32] = mag
        fp32_err[which, :, :, 1:, 32:] = mag
    bound = _bf16_ulp(want) + 2.0 ** -22 * fp32_err
    err = (planes.double() - want).abs()
    report(f"qkv rope {rope} b={b} n={n}: worst {(err / _bf16_ulp(want)).max().item():.2f} ulp")
    assert not torch.isnan(planes).any()
    assert (err <= bound).all(), (err / bound).max().item()
    assert torch.equal(planes[2], acc[2].float().to(BF))  # v and the cls rows are not rotated
    assert torch.equal(planes[:2, :, :, 0], acc[:2, :, :, 0].float().to(BF))


@pytest.mark.parametrize("with_pos", [False, True])
def test_patch_embed_integer_many_units(with_pos):
    """PatchEmbedEpi2 at 224 px, P 16, E 768, batch 128 (~4 units per cluster): integer images and weights, a bf16 bias
    off the integer grid; fp32 tokens = bf16(acc + bias) (+ pos) bit for bit, cls rows = cls_token."""
    lib = _lib.load()
    bsz, c, hw, p, e = 128, 3, 224, 16, 768
    np_ = (hw // p) ** 2
    assert _tiles(bsz * np_, e) >= 2 * _clusters()
    img = _ints((bsz, c, hw, hw), 3, seed=51).float()
    w = _ints((e, c, p, p), 3, seed=52)
    bias = _off_grid_bias(e).to(BF)
    g = torch.Generator(device=DEV).manual_seed(53)
    cls = torch.randn(e, generator=g, device=DEV)
    pos = torch.randn(np_, e, generator=g, device=DEV) if with_pos else None
    tok = torch.full((bsz, np_ + 1, e), NAN, device=DEV)
    ws_bytes = lib.vrr_patch_embed_workspace_bytes(bsz, c, hw, hw, p, e, _lib.VRR_BF16)
    ws = torch.empty(ws_bytes, device=DEV, dtype=torch.uint8)
    with tcgen05_must_run():
        _lib.check(lib.vrr_patch_embed_fwd(_p(img), _p(w), _p(bias), _p(cls), _p(pos), _p(tok), _p(ws), ws_bytes, bsz, c,
                                           hw, hw, p, e, _lib.VRR_F32, _lib.VRR_BF16, _lib.VRR_F32, _st()), "patch_embed")
    cols = F.unfold(img.double(), p, stride=p).transpose(1, 2)  # [B, Np, C P P]
    acc = (cols @ w.double().reshape(e, -1).t()).float()
    want = (acc + bias.float()).to(BF).float()
    if with_pos:
        want = want + pos
    got = tok[:, 1:].reshape(bsz * np_, e)
    assert _mismatch(got, want.reshape(bsz * np_, e), e) is None
    assert torch.equal(tok[:, 0], cls.expand(bsz, e))


# ------------------------------------------------------------------------------------- C: attention

SCALE = 64 ** -0.5


def _bias_case(kind, h, n, seed=0):
    """(vrr_bias_desc or None, fp32 parameter on the device, float64 bias [H][N][N] on the device)."""
    g = torch.Generator().manual_seed(seed + 5)
    if kind == "none":
        return None, None, None
    if kind == "table":
        tab = (torch.randn(h, 2 * n - 1, generator=g) * 0.5).to(DEV)
        idx = torch.arange(n, device=DEV)
        rel = idx[:, None] - idx[None, :] + n - 1
        return _lib.BiasDesc(_lib.BIAS_TABLE, h, 2 * n - 1, 0, tab.data_ptr()), tab, tab.double()[:, rel]
    grid = int(round((n - 1) ** 0.5))
    span = torch.tensor([float(max(2 * grid - 2, 1)) ** -kk for kk in range(4)])  # keeps |bias| O(1)
    coef = ((torch.randn(4, generator=g) if kind == "poly" else torch.randn(h, 4, generator=g)) * 0.7 * span).to(DEV)
    d = torch.zeros(n, n, dtype=torch.float64, device=DEV)
    d[1:, 1:] = torch.from_numpy(T.poly_l1_distance(n - 1)).double().to(DEV)
    pw = torch.stack([d ** kk for kk in range(4)], -1)  # [N, N, 4]
    pw[0, :, :] = 0.0
    pw[:, 0, :] = 0.0
    c2 = coef.double().view(-1, 4)
    bias = torch.einsum("ijk,hk->hij", pw, c2).expand(h, n, n)
    heads = 1 if kind == "poly" else h
    return _lib.BiasDesc(_lib.BIAS_POLY, heads, 4, grid, coef.data_ptr()), coef, bias


def _ref(planes, bias64, d_out=None, out=None):
    """float64 attention (the formulas of oracle/attention_np.py) on the device; the backward takes delta from the
    STORED output, as the kernels do."""
    b, h, n = planes.shape[1], planes.shape[2], planes.shape[3]
    q, k, v = planes.double().unbind(0)
    s = q @ k.transpose(-1, -2) * SCALE
    if bias64 is not None:
        s = s + bias64[None]
    lse = torch.logsumexp(s, -1)
    p = torch.exp(s - lse[..., None])
    o = p @ v
    if d_out is None:
        return o, lse
    do = d_out.double().view(b, n, h, 64).permute(0, 2, 1, 3)
    ob = out.double().view(b, n, h, 64).permute(0, 2, 1, 3)
    ds = p * (do @ v.transpose(-1, -2) - (do * ob).sum(-1, keepdim=True))
    grads = torch.stack([ds @ k * SCALE, ds.transpose(-1, -2) @ q * SCALE, p.transpose(-1, -2) @ do])
    return o, lse, grads, ds.sum(0)


def _dparam_ref(kind, dbias, n):
    if kind == "table":
        idx = torch.arange(n, device=DEV)
        rel = (idx[:, None] - idx[None, :] + n - 1).flatten()
        return torch.zeros(dbias.shape[0], 2 * n - 1, dtype=torch.float64, device=DEV).index_add_(1, rel, dbias.flatten(1))
    d = torch.zeros(n, n, dtype=torch.float64, device=DEV)
    d[1:, 1:] = torch.from_numpy(T.poly_l1_distance(n - 1)).double().to(DEV)
    mask = torch.zeros(n, n, dtype=torch.float64, device=DEV)
    mask[1:, 1:] = 1.0
    per_head = torch.stack([(dbias * mask * d ** kk).sum((1, 2)) for kk in range(4)], -1)  # [H, 4]
    return per_head.sum(0) if kind == "poly" else per_head


def _planes(b, h, n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.randn(3, b, h, n, 64, generator=g, device=DEV) * 0.8).to(BF)


def _fwd(planes, desc, dtype=_lib.VRR_BF16):
    _, b, h, n, dh = planes.shape
    out = torch.full((b, n, h * dh), NAN, device=DEV, dtype=planes.dtype)
    lse = torch.full((b, h, n), NAN, device=DEV)
    _lib.check(_lib.load().vrr_attn_fwd(_p(planes), None if desc is None else ctypes.byref(desc), _p(out), _p(lse), b, h,
                                        n, dh, ctypes.c_float(dh ** -0.5), dtype, _st()), "attn_fwd")
    return out, lse


def _bwd(planes, desc, param, out, d_out, lse):
    lib = _lib.load()
    _, b, h, n, _ = planes.shape
    dref = None if desc is None else ctypes.byref(desc)
    ws_bytes = lib.vrr_attn_bwd_workspace_bytes(b, h, n, 64, dref)
    ws = torch.empty(ws_bytes, device=DEV, dtype=torch.uint8)
    d_planes = torch.full_like(planes, NAN)
    d_param = None if param is None else torch.full_like(param, NAN)
    _lib.check(lib.vrr_attn_bwd(_p(planes), dref, _p(out), _p(d_out), _p(lse), _p(d_planes), _p(d_param), _p(ws), ws_bytes,
                                b, h, n, 64, ctypes.c_float(SCALE), _lib.VRR_BF16, _st()), "attn_bwd")
    return d_planes, d_param


def _per_item(got, want, dims):
    return ((got.double() - want).abs().amax(dims) / want.abs().amax(dims).clamp_min(1e-6))


def _check_attention(kind, b, h, n, seed):
    desc, param, bias64 = _bias_case(kind, h, n, seed)
    planes = _planes(b, h, n, seed)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    d_out = (torch.randn(b, n, h * 64, generator=g, device=DEV) * 0.5).to(BF)
    with tcgen05_must_run():
        out, lse = _fwd(planes, desc)
        d_planes, d_param = _bwd(planes, desc, param, out, d_out, lse)
    o, lse_ref, grads, dbias = _ref(planes, bias64, d_out, out)
    e_out = _per_item(out.view(b, n, h, 64).permute(0, 2, 1, 3), o, (2, 3))
    e_lse = ((lse.double() - lse_ref).abs() / lse_ref.abs().clamp_min(1.0)).amax(2)
    e_grad = _per_item(d_planes, grads, (3, 4))
    tag = f"{kind} B={b} H={h} N={n}"
    report(f"attention {tag}: worst per-item out {e_out.max().item():.2e} lse {e_lse.max().item():.2e} "
           f"grad {e_grad.max().item():.2e}")
    assert not torch.isnan(out).any() and not torch.isnan(lse).any() and not torch.isnan(d_planes).any(), tag
    worst = lambda e: (np.unravel_index(int(e.argmax()), tuple(e.shape)), e.max().item())  # noqa: E731
    assert e_out.max().item() <= 2e-2, (tag, "out", worst(e_out))
    assert e_lse.max().item() <= 1e-3, (tag, "lse", worst(e_lse))
    assert e_grad.max().item() <= 4e-2, (tag, "d_planes", worst(e_grad))
    if param is not None:
        want = _dparam_ref(kind, dbias, n)
        dims = (1,) if want.dim() == 2 else (0,)
        e_p = _per_item(d_param.view_as(want), want, dims)
        report(f"attention {tag}: worst per-head d_param {e_p.max().item():.2e}")
        assert e_p.max().item() <= (2e-2 if kind == "table" else 4e-2), (tag, "d_param", e_p)


ATTN_AT_SCALE = ([("table", 12, 197), ("poly", 12, 197), ("poly_perhead", 12, 197)]
                 + [("table", 4, n) for n in (65, 128, 129, 256)]
                 + [(kind, 4, n) for n in (122, 145, 226) for kind in ("poly", "poly_perhead")])


@pytest.mark.parametrize("kind,h,n", ATTN_AT_SCALE)
def test_biased_attention_many_items_per_cta(kind, h, n):
    """Biased attention with B*H >= 3 x SM items (every CTA of the persistent forward walks >= 3 items: table row
    prefetched one item ahead, the last head's tail patch, the shared-coefficient LUT kept across items): out, lse
    and d_planes per item, d_table / d_coef per head against float64 torch on the device.  H >= 4, so every 16-byte
    alignment of a table row occurs."""
    b = -(-3 * _sms() // h)
    _check_attention(kind, b, h, n, seed=n + h)


@pytest.mark.parametrize("kind", ["none", "table"])
@pytest.mark.parametrize("n", [128, 129, 208, 209, 256, 257])
def test_attention_dispatch_boundaries(n, kind):
    """Either side of every threshold of the default dispatch: one -> two softmax groups (128 / 129), whole-sequence
    -> tiled backward (208 / 209), whole-sequence -> tiled forward (256 / 257); fwd + bwd vs float64."""
    _check_attention(kind, 2, 4, n, seed=n)


def _batch_invariance(kind, b, h, n):
    desc, param, _ = _bias_case(kind, h, n, seed=n)
    planes = _planes(b, h, n, seed=61)
    g = torch.Generator(device=DEV).manual_seed(62)
    d_out = (torch.randn(b, n, h * 64, generator=g, device=DEV) * 0.5).to(BF)
    with tcgen05_must_run():
        out, lse = _fwd(planes, desc)
        d_planes, _ = _bwd(planes, desc, param, out, d_out, lse)
        for img in (0, 1, b // 2, b - 1):
            one = planes[:, img:img + 1].contiguous()
            o1, l1 = _fwd(one, desc)
            assert torch.equal(o1[0], out[img]) and torch.equal(l1[0], lse[img]), ("forward", img)
            dp1, _ = _bwd(one, desc, param, out[img:img + 1].contiguous(), d_out[img:img + 1].contiguous(),
                          lse[img:img + 1].contiguous())
            assert torch.equal(dp1[:, 0], d_planes[:, img]), ("backward", img)


@pytest.mark.parametrize("kind,n", [
    ("table", 197),   # whole-sequence forward with a bias (attn_fwd_ws), two-kernel backward (attn_bwd_tc2)
    ("poly", 197),
    ("none", 197),    # four-CTA forward (attn_fwd_tc4), whole-sequence backward (attn_bwd_ws)
    ("table", 257),   # tiled forward with a bias (attn_fwd_tc2), attn_bwd_tc2
])
def test_attention_batch_invariance_bitwise(kind, n):
    """Image b's out, lse and d_planes computed inside a batch of B*H >= 3 x SM items equal, bit for bit, the same
    image computed alone: the forward kernels and dQ / dK / dV have no atomics, so any difference is cross-item
    contamination (a stale buffer, a wrong item index) that no tolerance would catch."""
    h = 12
    _batch_invariance(kind, -(-3 * _sms() // h), h, n)


LSE_CASES = [  # (bias kind, N): each tcgen05 forward kernel through the default dispatch
    ("none", 197), ("none", 257),     # attn_fwd_tc4_kernel
    ("table", 197),                   # attn_fwd_ws_kernel
    ("table", 257)]                   # attn_fwd_tc2_kernel


@pytest.mark.parametrize("kind,n", LSE_CASES)
def test_lse_every_tcgen05_forward(kind, n):
    """lse (natural log of sum exp of the scaled, biased logits, vrr.h) of every tcgen05 forward kernel, every row
    including those of the ragged last tile, against float64 logsumexp."""
    b, h = 3, 4
    desc, _, bias64 = _bias_case(kind, h, n, seed=5)
    planes = _planes(b, h, n, seed=71)
    with tcgen05_must_run():
        out, lse = _fwd(planes, desc)
    o, lse_ref = _ref(planes, bias64)
    e = ((lse.double() - lse_ref).abs() / lse_ref.abs().clamp_min(1.0)).max().item()
    assert e <= 1e-3, e
    assert (out.view(b, n, h, 64).permute(0, 2, 1, 3).double() - o).abs().max().item() <= 2e-2 * o.abs().max().item()


@pytest.mark.parametrize("dtype,dh", [(torch.float32, 64), (torch.bfloat16, 32), (torch.float32, 16)])
def test_lse_simt_forward(dtype, dh):
    """lse of the SIMT forward (fp32, or head dim != 64) against float64 logsumexp, with a relative-table bias."""
    b, h, n = 2, 3, 197
    g = torch.Generator(device=DEV).manual_seed(81)
    planes = (torch.randn(3, b, h, n, dh, generator=g, device=DEV) * 0.8).to(dtype)
    desc, _, bias64 = _bias_case("table", h, n, seed=3)
    simt0 = _lib.family_count(_lib.IMPL_SIMT)
    out, lse = _fwd(planes, desc, _lib.VRR_F32 if dtype == torch.float32 else _lib.VRR_BF16)
    assert _lib.family_count(_lib.IMPL_SIMT) == simt0 + 1
    q, k, _ = planes.double().unbind(0)
    lse_ref = torch.logsumexp(q @ k.transpose(-1, -2) * dh ** -0.5 + bias64[None], -1)
    e = ((lse.double() - lse_ref).abs() / lse_ref.abs().clamp_min(1.0)).max().item()
    assert e <= (1e-5 if dtype == torch.float32 else 1e-3), e
