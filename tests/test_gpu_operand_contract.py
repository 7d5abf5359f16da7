"""The GEMM operand producers of the model pass (pnp_ovss_b200/csrc/tf32x3.cu) against plain references, at production sizes
and at the edges of their contract: the plain splits (TF32 and 3xFP16), GELU + split, residual + LayerNorm + split, the
3xFP16 bias columns and the fp16 overflow flag.

Every GEMM of the ViT-L encoder and every text-side _Linear3 reads its left operand from one of these.  Splits are integer
work and compared bit for bit; GELU and LayerNorm are compared with fp64 within 2x torch's own fp32 error on the same input
(the maximum over a band of inputs or a kind of row), plus a stated floor.  Row generators and the reduction order of the
LayerNorm are in test_operand_algorithm.py."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_kernels import _split16_ref, _split_ref
from test_operand_algorithm import LN_KS, ROW_KINDS, ln_mixed, ln_rows

pytestmark = pytest.mark.gpu

SPLIT_GRID = 148 * 16           # CTAs of the split kernels; each walks rows, 1024 columns per pass
LN_ROWS = 148 * 8 * 8           # rows the LayerNorm grid covers in one wave (CTAs x warps)
FP16_MAX = 65504.0
TF32_CARRY_OUT = float(np.array(0x7F7FF000, np.uint32).view(np.float32))   # rounds up to inf at bit 13


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ops():
    from pnp_ovss_b200 import ops as _ops
    return _ops


@pytest.fixture(scope="module")
def lib():
    from pnp_ovss_b200 import _lib
    return _lib.load()


def _flag(dev, value=0):
    return torch.full((1,), value, dtype=torch.int32, device=dev)


def _same_bits(got, want):
    """Bit-equal, except that a NaN only has to be a NaN (payloads differ between the device and torch)."""
    assert got.shape == want.shape and got.dtype == want.dtype
    assert torch.equal(got.isnan(), want.isnan())
    ok = ~want.isnan()
    assert torch.equal(got[ok], want[ok])


def _tf32_split_ieee(t):
    """_split_ref extended past the finite range: where rounding would carry past the largest finite value (|x| from
    0x7F7FF000 up, +-inf, NaN) hi = x and lo = 0, or NaN for a NaN x.  _split_ref gives inf - inf there, and rounds the
    arithmetic NaN 0x7FFFFFFF to -0, its carry landing in the sign bit."""
    hi = ((t.view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)
    hi = torch.where(t.abs() < TF32_CARRY_OUT, hi, t)
    lo = torch.where(hi == t, torch.zeros_like(t), t - hi)
    return torch.cat([hi, lo, hi], -1)


def _fp16_back(s3, K):
    """h + l 2^-11 in fp64 from a [h s | l | h] operand."""
    return s3[..., 2 * K:3 * K].double() + s3[..., K:2 * K].double() / 2048.0


def _within_reconstruction(back, x):
    # h + l 2^-11 carries 22-23 bits; below fp16's normal range (2^-14) l is rounded to the subnormal spacing 2^-24, which
    # the 2^-11 scales to an absolute 2^-35 step: floor 2^-36
    return bool(((back - x.double()).abs() <= 2.0 ** -21 * x.double().abs() + 2.0 ** -36).all())


# ------------------------------------------------------------------------------------------------ plain splits
@pytest.mark.parametrize("M", [1, SPLIT_GRID + 1, 15470])
@pytest.mark.parametrize("K", [4, 8, 12, 1020, 1028, 3072, 4092, 4100])
def test_split_shapes(dev, ops, M, K):
    """K off and past the 1024-column pass of a CTA, M one row past the grid and at configs[1]'s ViT rows (35 x 442)."""
    g = torch.Generator(device=dev).manual_seed(M * 7 + K)
    x = torch.randn(M, K, generator=g, device=dev) * 3
    assert torch.equal(ops.tf32_split3(x), _split_ref(x))
    flag = _flag(dev)
    got = ops.fp16_split3(x, 1.0, 1.0, flag)
    assert torch.equal(got, _split16_ref(x)) and int(flag.item()) == 0
    assert _within_reconstruction(_fp16_back(got, K), x)


def test_tf32_ties_round_away_from_zero(dev, ops):
    """Bits 0-12 exactly 0x1000 are a tie at TF32's last mantissa bit (bit 13): the magnitude rounds up whether bit 13 is even
    or odd, and may carry into the exponent."""
    base = np.array([0x3F800000, 0x3F802000, 0x3FFFE000, 0x00800000, 0x7F000000, 0x4B3FE000], np.uint32)
    mag = base | np.uint32(0x1000)
    want_mag = (mag & np.uint32(0xFFFFE000)) + np.uint32(0x2000)
    sign = np.uint32(0x80000000)
    x = torch.from_numpy(np.concatenate([mag, mag | sign, mag[:4]]).view(np.float32)).view(4, 4).to(dev)         # K = 4
    want = torch.from_numpy(np.concatenate([want_mag, want_mag | sign, want_mag[:4]]).view(np.float32)).view(4, 4).to(dev)
    got = ops.tf32_split3(x)
    assert torch.equal(got[:, :4], want) and torch.equal(got[:, 8:], want)
    assert torch.equal(got[:, :4] + got[:, 4:8], x)
    assert bool((want.abs() > x.abs()).all())                       # away from zero, also for the even bit 13
    assert float(want[0, 2]) == 2.0                               # 0x3FFFF000 carries into the exponent


SPECIALS = [0.0, -0.0, 1e-45, -1e-45, 1e-40, -2.0 ** -127, 2.0 ** -126, 3e-8, -2.0 ** -25, 2.0 ** -24, 1e-5, -6e-5,
            2.0 ** -14 * (1 - 2.0 ** -12), 2.0 ** -14, 1.0 + 2.0 ** -23, -3.0]


def test_split_subnormals_and_zeros(dev, ops):
    x = torch.tensor(SPECIALS, device=dev).view(2, 8)
    assert torch.equal(ops.tf32_split3(x).view(torch.int32), _tf32_split_ieee(x).view(torch.int32))     # -0 stays -0
    flag = _flag(dev)
    got = ops.fp16_split3(x, 1.0, 1.0, flag)
    assert torch.equal(got.view(torch.int16), _split16_ref(x).view(torch.int16)) and int(flag.item()) == 0
    assert _within_reconstruction(_fp16_back(got, 8), x)
    tiny = torch.randn(64, 1024, generator=torch.Generator(device=dev).manual_seed(3), device=dev)
    for scale in (2.0 ** -14, 2.0 ** -20, 2.0 ** -30):
        got = ops.fp16_split3(tiny * scale, 1.0, 1.0, flag)
        assert torch.equal(got, _split16_ref(tiny * scale)) and _within_reconstruction(_fp16_back(got, 1024), tiny * scale)
    assert int(flag.item()) == 0


def test_split_infinities_and_nan(dev, ops):
    """TF32: hi = x and lo = 0 for +-inf and for finite values whose rounding would overflow; NaN stays NaN.  fp16: the torch
    restatement's h and l (l = NaN for inf), and the flag."""
    fmax = float(np.finfo(np.float32).max)
    below = float(np.nextafter(np.float32(TF32_CARRY_OUT), np.float32(0)))
    x = torch.tensor([[float("inf"), -float("inf"), fmax, -TF32_CARRY_OUT], [float("nan"), 1.0, -0.0, -below]], device=dev)
    x[1, 1] = x[1, 1] * float("nan")                           # the device's arithmetic NaN, 0x7FFFFFFF
    got = ops.tf32_split3(x)
    _same_bits(got, _tf32_split_ieee(x))
    assert torch.equal(got[0, :4], x[0]) and not got[0, 4:8].any()
    assert bool(got[1, :2].isnan().all()) and bool(got[1, 8:10].isnan().all())    # NaN stays NaN in hi, not -0
    assert float(got[1, 3]) == -(TF32_CARRY_OUT - 2.0 ** 116) and float(got[1, 3] + got[1, 7]) == -below
    for row in range(2):
        flag = _flag(dev)
        got = ops.fp16_split3(x[row:row + 1].contiguous(), 1.0, 1.0, flag)
        _same_bits(got, _split16_ref(x[row:row + 1]))
        assert int(flag.item()) == 1


@pytest.mark.parametrize("hi_scale", [1.0, 4.0])
def test_fp16_flag_at_the_rounding_boundary(dev, ops, hi_scale):
    """The flag means: h * hi_scale, in fp16, is not finite.  An x that rounds to h = 65504 / hi_scale passes and is split
    exactly; the halfway point above rounds h up (ties to even) and overflows once scaled."""
    top = FP16_MAX / hi_scale
    half_step = 16.0 / hi_scale                                 # half the fp16 spacing at top: 16 at 65504, 4 at 16376
    exact = top + half_step - 0.5                               # (x - h) 2^11 is an fp16 number: exact reconstruction
    below = float(np.nextafter(np.float32(top + half_step), np.float32(0)))
    for sign in (1.0, -1.0):
        x = torch.tensor([[sign * exact, sign * below, 1.0, -2.0]], device=dev)
        flag = _flag(dev)
        got = ops.fp16_split3(x, 1.0, hi_scale, flag)
        assert int(flag.item()) == 0, (sign, hi_scale)
        assert float(got[0, 0]) == sign * FP16_MAX and float(got[0, 1]) == sign * FP16_MAX
        back = _fp16_back(got, 4)
        assert float(back[0, 0]) == sign * exact and _within_reconstruction(back, x)
        assert torch.equal(got, _split16_ref(x, hi_scale))
        over = torch.tensor([[sign * (top + half_step), 1.0, 1.0, 1.0]], device=dev)
        ops.fp16_split3(over, 1.0, hi_scale, flag)
        assert int(flag.item()) == 1, (sign, hi_scale)


# ------------------------------------------------------------------------------------------------ overflow flag, every producer
def _ln_inputs(dev, K=1024, M=6, seed=0):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(M, K, generator=g, device=dev)
    gamma, beta = torch.randn(K, generator=g, device=dev), torch.randn(K, generator=g, device=dev)
    return x, gamma, beta


def _produce(ops, producer, x, flag, gamma=None, beta=None, split=True):
    if producer == "split":
        return ops.fp16_split3(x, 1.0, 1.0, flag)
    if producer == "gelu":
        return ops.gelu_fp16_split3(x, None, 1.0, 1.0, flag)
    return ops.layernorm_fp16_split3(x, gamma, beta, 1e-6, flag=flag, split=split, plain=not split,
                                     bias_one=64.0 if producer == "ln_bias" else None)[0]


@pytest.mark.parametrize("bad", ["nan", "inf", "-inf", "range"])
@pytest.mark.parametrize("producer", ["split", "gelu", "ln", "ln_bias"])
def test_flag_for_every_producer(dev, ops, producer, bad):
    """NaN or +-inf anywhere in a late row, or a value past fp16's range (70000 for the split and GELU; for the LayerNorm an
    output pushed to ~6e5 by one gamma) raises the flag; the same call without it does not; a raised flag is never cleared."""
    x, gamma, beta = _ln_inputs(dev)
    flag = _flag(dev)
    _produce(ops, producer, x, flag, gamma, beta)
    assert int(flag.item()) == 0
    preset = _flag(dev, 1)
    _produce(ops, producer, x, preset, gamma, beta)
    assert int(preset.item()) == 1
    xb, gb = x.clone(), gamma.clone()
    if bad == "range":
        if producer.startswith("ln"):
            xb[5, 1000] = 40.0                                    # ~ +10 sd after normalisation
            gb[1000] = 60000.0
        else:
            xb[5, 1000] = 70000.0
    else:
        xb[5, 1000] = float(bad)
    _produce(ops, producer, xb, flag, gb, beta)
    assert int(flag.item()) == 1


@pytest.mark.parametrize("bad", ["nan", "inf", "range"])
def test_ln_plain_output_never_raises_the_flag(dev, ops, bad):
    x, gamma, beta = _ln_inputs(dev)
    x[5, 1000], gamma[1000] = (40.0, 60000.0) if bad == "range" else (float(bad), gamma[1000])
    flag = _flag(dev)
    _, plain = ops.layernorm_fp16_split3(x, gamma, beta, 1e-6, split=False, plain=True, flag=flag)
    assert int(flag.item()) == 0
    assert float(plain[5].abs().max()) > FP16_MAX if bad == "range" else bool(plain[5].isnan().all())


def test_gelu_of_a_large_input_with_hi_scale(dev, ops):
    """GELU(x) = x for large x: 20000 fits fp16 but not once scaled by 4."""
    x = torch.full((2, 8), 1.0, device=dev)
    x[1, 3] = 20000.0
    flag = _flag(dev)
    ops.gelu_fp16_split3(x, None, 1.0, 1.0, flag)
    assert int(flag.item()) == 0
    ops.gelu_fp16_split3(x, None, 1.0, 4.0, flag)
    assert int(flag.item()) == 1


# ------------------------------------------------------------------------------------------------ GELU
GELU_BANDS = (-12.0, -10.0, -5.0, -1.0, 1.0, 5.0, 12.0)


def _assert_gelu_grade(back, v, is_fp16):
    """Per band of v: max |error| within 2x torch's fp32 gelu error against fp64, plus a floor of one fp32 rounding of
    erf near -1 (2^-24) times the 0.5 |v| in front of it, and for the fp16 form its reconstruction (2^-21 |y| + 2^-36)."""
    want = F.gelu(v.double())
    terr = (F.gelu(v).double() - want).abs()
    err = (back - want).abs()
    for lo, hi in zip(GELU_BANDS[:-1], GELU_BANDS[1:]):
        band = (v >= lo) & (v < hi)
        assert bool(band.any())
        floor = 2.0 ** -24 * 0.5 * float(v[band].abs().max())
        if is_fp16:
            floor += 2.0 ** -21 * float(want[band].abs().max()) + 2.0 ** -36
        assert float(err[band].max()) <= 2 * float(terr[band].max()) + floor, (lo, hi, float(err[band].max()), float(terr[band].max()))


@pytest.mark.parametrize("with_bias", [False, True])
def test_gelu_from_minus_12_to_12(dev, ops, with_bias):
    """Inputs across [-12, 12], the -10..-5 band where 1 + erf cancels included; with_bias: the production form, the input
    scaled by 2^11 and taken back by in_scale = 2^-11, a bias added."""
    M, K = 64, 4100
    v0 = torch.linspace(-12.0, 12.0, M * K, device=dev).view(M, K)
    bias = torch.randn(K, generator=torch.Generator(device=dev).manual_seed(5), device=dev) * 0.5 if with_bias else None
    v = v0 + bias if with_bias else v0
    x, in_scale = (v0 * 2048.0, 2.0 ** -11) if with_bias else (v0, 1.0)
    t3 = ops.gelu_tf32_split3(v0, bias) if with_bias else ops.gelu_tf32_split3(v0)
    y = t3[:, :K] + t3[:, K:2 * K]
    assert torch.equal(t3, _split_ref(y))
    _assert_gelu_grade(y.double(), v, False)
    flag = _flag(dev)
    h3 = ops.gelu_fp16_split3(x, bias, in_scale, 1.0, flag)
    assert int(flag.item()) == 0
    _assert_gelu_grade(_fp16_back(h3, K), v, True)


# ------------------------------------------------------------------------------------------------ LayerNorm
def _assert_ln_grade(got, x, gamma, beta, eps, kinds):
    """Per kind of row: max |error| against fp64 within 2x torch's fp32 layer_norm error on the same rows, plus a floor of
    2^-22 of the largest |y| (the final rounding of y = n gamma + beta)."""
    K = x.shape[-1]
    want = F.layer_norm(x.double(), (K,), gamma.double(), beta.double(), eps)
    terr = (F.layer_norm(x, (K,), gamma, beta, eps).double() - want).abs()
    err = (got.double() - want).abs()
    for i in kinds.unique().tolist():
        rows = kinds == i
        bound = 2 * float(terr[rows].max()) + 2.0 ** -22 * float(want[rows].abs().max())
        assert float(err[rows].max()) <= bound, (ROW_KINDS[i], float(err[rows].max()), float(terr[rows].max()))


def _ln_case(dev, M, K, seed):
    x, kinds = ln_mixed(M, K, seed)
    g = torch.Generator(device=dev).manual_seed(seed)
    gamma, beta = torch.randn(K, generator=g, device=dev), torch.randn(K, generator=g, device=dev)
    return torch.from_numpy(x).to(dev), torch.from_numpy(kinds).to(dev), gamma, beta


def _ln(ops, form, x, gamma, beta, eps, hi_scale=1.0, **kw):
    if form == "tf32":
        return ops.layernorm_tf32_split3(x, gamma, beta, eps, split=True, plain=True, **kw)
    flag = _flag(x.device)
    s3, plain = ops.layernorm_fp16_split3(x, gamma, beta, eps, hi_scale=hi_scale, split=True, plain=True, flag=flag, **kw)
    assert int(flag.item()) == 0
    return s3, plain


def _split_of(form, plain, hi_scale=1.0):
    return _split_ref(plain) if form == "tf32" else _split16_ref(plain, hi_scale)


@pytest.mark.parametrize("K", LN_KS)
@pytest.mark.parametrize("form", ["tf32", "fp16"])
def test_layernorm_row_kinds(dev, ops, form, K):
    """randn, large-offset, outlier-channel and constant rows at every template (6 / 8 / 16 chunks), full and partial."""
    x, kinds, gamma, beta = _ln_case(dev, 333, K, K)
    s3, plain = _ln(ops, form, x, gamma, beta, 1e-6)
    _assert_ln_grade(plain, x, gamma, beta, 1e-6, kinds)
    assert torch.equal(s3, _split_of(form, plain))


@pytest.mark.parametrize("K", LN_KS)
@pytest.mark.parametrize("eps", [1e-6, 1e-5])
@pytest.mark.parametrize("form", ["tf32", "fp16"])
def test_layernorm_constant_rows_give_beta(dev, ops, form, eps, K):
    """A constant row normalises to exactly 0, so y = beta, as torch's fp32 layer_norm gives; a mean rounded to fp32 without
    the correction, times rsqrt(eps), does not."""
    x = torch.from_numpy(ln_rows("constant", 24, K, 0)).to(dev)
    g = torch.Generator(device=dev).manual_seed(K)
    gamma, beta = torch.randn(K, generator=g, device=dev), torch.randn(K, generator=g, device=dev)
    s3, plain = _ln(ops, form, x, gamma, beta, eps)
    assert torch.equal(plain, beta.expand_as(plain))
    assert torch.equal(s3, _split_of(form, plain))


@pytest.mark.parametrize("M", [LN_ROWS + 1, 15470])
@pytest.mark.parametrize("form", ["tf32", "fp16"])
def test_layernorm_rows_beyond_one_wave(dev, ops, form, M):
    x, kinds, gamma, beta = _ln_case(dev, M, 1024, M)
    s3, plain = _ln(ops, form, x, gamma, beta, 1e-6)
    _assert_ln_grade(plain, x, gamma, beta, 1e-6, kinds)
    assert torch.equal(s3, _split_of(form, plain))


@pytest.mark.parametrize("with_bias", [False, True])
@pytest.mark.parametrize("scale", [1.0, 2.0 ** -11])
@pytest.mark.parametrize("form", ["tf32", "fp16"])
def test_layernorm_with_residual(dev, ops, form, scale, with_bias):
    """x <- x + residual * scale (+ bias), written back in place, then the LayerNorm of it (the TF32 form has scale 1 only)."""
    if form == "tf32" and scale != 1.0:
        pytest.skip("pnp_layernorm_tf32_split3 has no residual scale")
    x, kinds, gamma, beta = _ln_case(dev, 333, 1024, 17)
    g = torch.Generator(device=dev).manual_seed(18)
    res = torch.randn(x.shape, generator=g, device=dev) / scale
    rb = torch.randn(1024, generator=g, device=dev) if with_bias else None
    kw = dict(residual=res, residual_bias=rb) if form == "tf32" else dict(residual=res, residual_scale=scale, residual_bias=rb)
    xin = x.clone()
    s3, plain = _ln(ops, form, xin, gamma, beta, 1e-6, **kw)
    want_x = x + res * scale                                      # res * scale is exact: one rounding, as the kernel's fma
    if with_bias:
        want_x = want_x + rb
    assert torch.equal(xin, want_x)
    _assert_ln_grade(plain, xin, gamma, beta, 1e-6, kinds)
    assert torch.equal(s3, _split_of(form, plain))


def _abi_ln(lib, form, x, res, x_out, gamma, beta, out3, out1, ld3=None, bias_one=0.0, hi_scale=1.0, flag=None, scale=1.0):
    M, K = x.shape
    p = lambda t: None if t is None else t.data_ptr()
    if form == "tf32":
        return lib.pnp_layernorm_tf32_split3(p(x), p(res), None, p(x_out), p(gamma), p(beta), 1e-6, p(out3), p(out1), M, K, None)
    return lib.pnp_layernorm_fp16_split3(p(x), p(res), scale, None, p(x_out), p(gamma), p(beta), 1e-6, hi_scale, p(out3),
                                         3 * K if ld3 is None else ld3, bias_one, p(out1), p(flag), M, K, None)


@pytest.mark.parametrize("form", ["tf32", "fp16"])
def test_layernorm_x_out_in_place_separate_or_null(dev, lib, form):
    """With a residual, x_out may alias x, be a buffer of its own (x is then left alone) or be NULL (nothing written back):
    the LayerNorm and its split are the same in all three."""
    x, _, gamma, beta = _ln_case(dev, 333, 1024, 23)
    res = torch.randn(x.shape, generator=torch.Generator(device=dev).manual_seed(24), device=dev)
    want_x = x + res
    dtype = torch.float32 if form == "tf32" else torch.float16
    outs = []
    for mode in ("in_place", "separate", "null"):
        xin = x.clone()
        x_out = {"in_place": xin, "separate": torch.full_like(x, float("nan")), "null": None}[mode]
        out3, out1 = torch.full((333, 3 * 1024), float("nan"), dtype=dtype, device=dev), torch.full_like(x, float("nan"))
        assert _abi_ln(lib, form, xin, res, x_out, gamma, beta, out3, out1) == 0
        torch.cuda.synchronize()
        if mode == "separate":
            assert torch.equal(x_out, want_x) and torch.equal(xin, x)
        else:
            assert torch.equal(xin, want_x if mode == "in_place" else x)
        outs.append((out3, out1))
    for out3, out1 in outs[1:]:
        assert torch.equal(out3, outs[0][0]) and torch.equal(out1, outs[0][1])
    assert torch.equal(outs[0][0], _split_of(form, outs[0][1]))


# ------------------------------------------------------------------------------------------------ bias columns
@pytest.mark.parametrize("hi_scale", [1.0, 4.0])
@pytest.mark.parametrize("K", [768, 1024])
def test_bias_columns_on_every_row(dev, lib, K, hi_scale):
    """ld_out3 = 3K + 8: every row, odd and even, ends in [bias_one, 1, 0 x 6] and starts with the split of the plain output;
    the output is NaN-filled first, so an unwritten cell shows."""
    M = LN_ROWS + 1
    x, _, gamma, beta = _ln_case(dev, M, K, K + 1)
    out3 = torch.full((M, 3 * K + 8), float("nan"), dtype=torch.float16, device=dev)
    out1 = torch.full_like(x, float("nan"))
    flag = _flag(dev)
    assert _abi_ln(lib, "fp16", x, None, None, gamma, beta, out3, out1, ld3=3 * K + 8, bias_one=64.0, hi_scale=hi_scale, flag=flag) == 0
    tail = torch.tensor([64.0, 1.0, 0, 0, 0, 0, 0, 0], dtype=torch.float16, device=dev).expand(M, 8)
    assert torch.equal(out3[:, 3 * K:].view(torch.int16), tail.view(torch.int16))   # +0, not -0, in the zero columns
    assert torch.equal(out3[:, :3 * K], _split16_ref(out1, hi_scale)) and int(flag.item()) == 0


def test_bias_columns_end_to_end(dev, ops):
    """_mm16(LayerNorm split with bias columns, _w16(W, b)) / 2^11 = LN(x) W^T + b at the fp32-grade bound of
    test_tripled_fp16_gemm_is_fp32_grade."""
    from pnp_ovss_b200.blip_itm import FP16_BIAS_ONE, FP16_OUT_SCALE, _mm16, _w16
    g = torch.Generator(device=dev).manual_seed(31)
    x = torch.randn(512, 1024, generator=g, device=dev) * 2 + 0.3
    gamma, beta = torch.randn(1024, generator=g, device=dev), torch.randn(1024, generator=g, device=dev)
    w, b = torch.randn(768, 1024, generator=g, device=dev) * 0.02, torch.randn(768, generator=g, device=dev)
    w16, hi_scale = _w16(w, b)
    s3, plain = ops.layernorm_fp16_split3(x, gamma, beta, 1e-6, hi_scale=hi_scale, plain=True, bias_one=FP16_BIAS_ONE)
    y = _mm16(s3, w16) / FP16_OUT_SCALE
    truth = F.linear(F.layer_norm(x.double(), (1024,), gamma.double(), beta.double(), 1e-6), w.double(), b.double())
    err3 = (y.double() - truth).abs().max().item()
    err32 = (F.linear(plain, w, b).double() - truth).abs().max().item()
    assert err3 <= 12 * err32 + 1e-6, (err3, err32)


@pytest.mark.parametrize("K", [12, 1020])
def test_bias_columns_refuse_k_not_a_multiple_of_8(dev, ops, lib, K):
    """The 8 bias columns of a row are one 16-byte store at half offset m (3K + 8) + 3K, which is 16-byte aligned for
    every row only when K % 8 == 0: the wrapper raises and the ABI returns -1 before any launch."""
    from pnp_ovss_b200 import PnpError
    M = 5
    x, gamma, beta = _ln_inputs(dev, K=K, M=M)
    with pytest.raises(PnpError):
        ops.layernorm_fp16_split3(x, gamma, beta, 1e-6, bias_one=64.0)
    out3 = torch.full((M, 3 * K + 8), float("nan"), dtype=torch.float16, device=dev)
    assert _abi_ln(lib, "fp16", x, None, None, gamma, beta, out3, None, ld3=3 * K + 8, bias_one=64.0) == -1
    torch.cuda.synchronize()
    assert bool(out3.isnan().all())
    s3, _ = ops.layernorm_fp16_split3(x, gamma, beta, 1e-6)          # the same K without bias columns is fine
    assert s3.shape == (M, 3 * K)
