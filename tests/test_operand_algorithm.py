"""The LayerNorm reduction order of layernorm_split3_kernel and the algebra of the 3xFP16 bias columns, restated on the CPU
(pnp_ovss_b200/csrc/tf32x3.cu, pnp_ovss_b200/blip_itm.py).  test_gpu_operand_contract.py holds the kernels to these and
builds its inputs with the row generators below.

One warp normalises one row.  Lane l holds the float4 chunks k = 4 (l + 32 c), c < ceil(K / 128); it sums each chunk as
(x0 + x1) + (x2 + x3) onto a running fp32 sum, and the 32 lane sums meet in an xor butterfly (warp_sum).  The kernel takes the
mean m0 = sum / K, then a second pass over the deviations v - m0: it sums their squares and, since the corrected two-pass
form, the deviations themselves, whose mean r moves the mean to m0 + r and takes r^2 out of the variance.  The plain order
multiplies m0's rounding error by rsqrt(var + eps), about rsqrt(eps) on a constant row.  The restatement does not model the
device's FMA contraction or its rsqrtf: it reproduces the regimes, not the last bit."""
import numpy as np
import pytest
import torch

from pnp_ovss_b200.blip_itm import FP16_BIAS_ONE, FP16_OUT_SCALE, _w16

f32 = np.float32
LN_KS = (4, 124, 128, 132, 764, 768, 772, 1020, 1024, 1028, 2044, 2048)   # every template, full and partial last chunks
ROW_KINDS = ("randn", "offset", "outlier", "constant")
CONSTANTS = (0.3, 1.7, -2.3, 100.1, 0.1, 3.0)


def ln_rows(kind, M, K, seed):
    """[M, K] float32 rows of one kind: randn (2 N + 0.3), offset (1000 + 0.1 N: the variance is 1e-8 of E[x^2]),
    outlier (N with four ViT-L-style channels at +-500), constant (one of CONSTANTS per row)."""
    rng = np.random.default_rng(seed)
    if kind == "randn":
        x = 2.0 * rng.standard_normal((M, K)) + 0.3
    elif kind == "offset":
        x = 1000.0 + 0.1 * rng.standard_normal((M, K))
    elif kind == "outlier":
        x = rng.standard_normal((M, K))
        ch = rng.choice(K, size=min(4, K), replace=False)
        x[:, ch] = 500.0 * np.sign(rng.standard_normal((M, ch.size)))
    elif kind == "constant":
        x = np.repeat(np.asarray(CONSTANTS)[np.arange(M) % len(CONSTANTS), None], K, 1)
    else:
        raise ValueError(kind)
    return x.astype(f32)


def ln_mixed(M, K, seed):
    """M rows cycling through ROW_KINDS (row m is of kind m % 4), and the kind of each row."""
    kinds = np.arange(M) % len(ROW_KINDS)
    x = np.empty((M, K), f32)
    for i, kind in enumerate(ROW_KINDS):
        rows = np.flatnonzero(kinds == i)
        x[rows] = ln_rows(kind, rows.size, K, seed + i)
    return x, kinds


def _lane_chunks(x):
    """[M, K] -> [M, C, 32, 4] float32, chunk c of lane l = x[:, 4 (l + 32 c) : +4], zero past K; and its validity [C, 32]."""
    M, K = x.shape
    C = (K + 127) // 128
    pad = np.zeros((M, C * 128), f32)
    pad[:, :K] = x
    valid = (np.arange(C)[:, None] * 32 + np.arange(32)[None, :]) * 4 < K
    return pad.reshape(M, C, 32, 4), valid


def _lane_sums(parts, valid):
    s = np.zeros(parts.shape[::2], f32)             # [M, 32]
    for c in range(parts.shape[1]):
        s = np.where(valid[c], (s + parts[:, c]).astype(f32), s)
    return s


def _warp_sum(s):
    for o in (16, 8, 4, 2, 1):
        s = (s + s[:, np.arange(32) ^ o]).astype(f32)
    return s[:, 0]


def ln_moments(x, corrected=True):
    """(mean, var) float32 per row in the kernel's order; corrected=False: the plain two-pass form (mean m0, var around it)."""
    K = x.shape[1]
    t, valid = _lane_chunks(x)
    m0 = (_warp_sum(_lane_sums((t[..., 0] + t[..., 1]) + (t[..., 2] + t[..., 3]), valid)) / f32(K)).astype(f32)
    d = (t - m0[:, None, None, None]).astype(f32)
    sq = _warp_sum(_lane_sums((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + (d[..., 2] * d[..., 2] + d[..., 3] * d[..., 3]), valid))
    if not corrected:
        return m0, (sq / f32(K)).astype(f32)
    dev = _warp_sum(_lane_sums((d[..., 0] + d[..., 1]) + (d[..., 2] + d[..., 3]), valid))
    r = (dev / f32(K)).astype(f32)
    return (m0 + r).astype(f32), (np.maximum(sq - dev * r, f32(0)) / f32(K)).astype(f32)


def ln_restated(x, eps, corrected=True, one_pass=False):
    """(x - mean) * rstd in float32 (gamma 1, beta 0).  one_pass: variance as E[x^2] - mean^2 (a wrong kernel, for contrast)."""
    mean, var = ln_moments(x, corrected)
    if one_pass:
        var = np.maximum((x.astype(f32) ** 2).mean(1, dtype=f32) - mean * mean, 0).astype(f32)
    rstd = (1.0 / np.sqrt(var.astype(np.float64) + np.float64(f32(eps)))).astype(f32)
    return ((x - mean[:, None]) * rstd[:, None]).astype(f32)


def ln_exact(x, eps):
    x = x.astype(np.float64)
    m = x.mean(1, keepdims=True)
    return (x - m) / np.sqrt(((x - m) ** 2).mean(1, keepdims=True) + np.float64(f32(eps)))


def torch_ln_err(x, eps):
    want = ln_exact(x, eps)
    got = torch.nn.functional.layer_norm(torch.from_numpy(x), (x.shape[1],), eps=eps).double().numpy()
    return np.abs(got - want).max(1)


# ---------------------------------------------------------------------------------------------------- LayerNorm order
@pytest.mark.parametrize("c,K,err", [(0.3, 768, 3.0e-5), (1.7, 1024, 1.2e-4), (100.1, 1024, 7.6e-3)])
def test_constant_rows_show_the_mean_rounding_without_the_correction(c, K, err):
    x = np.full((1, K), c, f32)
    old = np.abs(ln_restated(x, 1e-6, corrected=False)).max()
    assert abs(old - err) <= 0.05 * err, old                    # the plain order: |y - beta| = err |gamma|
    assert not ln_restated(x, 1e-6).any()                       # corrected: exactly 0, as torch's fp32 layer_norm
    assert not torch.nn.functional.layer_norm(torch.from_numpy(x), (K,), eps=1e-6).any()


@pytest.mark.parametrize("K", LN_KS)
def test_corrected_order_is_exact_on_every_constant_row(K):
    x = ln_rows("constant", len(CONSTANTS), K, 0)
    for eps in (1e-6, 1e-5):
        assert not ln_restated(x, eps).any()


@pytest.mark.parametrize("K", LN_KS)
def test_constant_rows_reach_an_inexact_mean(K):
    """The GPU's constant rows test the correction only where m0 is not the row's value: at every K whose chunk sums are
    not all exact (not at K = 4 or 128, where every lane holds one chunk, 4 times the value, and the butterfly only doubles)."""
    x = ln_rows("constant", len(CONSTANTS), K, 0)
    m0, _ = ln_moments(x, corrected=False)
    inexact = m0 != x[:, 0]
    assert inexact.any() == (K not in (4, 128)), m0 - x[:, 0]
    if inexact.any():
        assert np.abs(ln_restated(x, 1e-6, corrected=False)).max() > 1e-6


@pytest.mark.parametrize("K", (764, 1024, 2044))
@pytest.mark.parametrize("kind", ("randn", "offset", "outlier"))
def test_corrected_order_is_as_good_as_torch(K, kind):
    """On rows with a spread the correction changes little; it stays within 2x torch's fp32 error (+ 2^-22 of the largest
    |y|), and so within the bound the GPU tests use."""
    x = ln_rows(kind, 64, K, K)
    want = ln_exact(x, 1e-6)
    err = np.abs(ln_restated(x, 1e-6) - want).max()
    assert err <= 2 * torch_ln_err(x, 1e-6).max() + 2.0 ** -22 * np.abs(want).max(), err


def test_offset_rows_catch_a_one_pass_variance():
    """1000 + 0.1 N: E[x^2] - mean^2 cancels 1e6 down to 1e-2 in fp32, so a one-pass variance misses by orders of magnitude."""
    x = ln_rows("offset", 16, 1024, 3)
    want = ln_exact(x, 1e-6)
    bound = 2 * torch_ln_err(x, 1e-6).max() + 2.0 ** -22 * np.abs(want).max()
    assert np.abs(ln_restated(x, 1e-6, one_pass=True) - want).max() > 100 * bound


def test_row_generators_reach_their_regimes():
    x, kinds = ln_mixed(333, 1028, 5)
    assert (np.bincount(kinds) >= 83).all()
    m0, var = ln_moments(x[kinds == 1], corrected=False)
    assert (np.abs(m0 - 1000) < 0.1).all() and (var < 0.02).all()
    out = x[kinds == 2]
    assert ((np.abs(out) == 500).sum(1) == 4).all()
    _, valid = _lane_chunks(np.zeros((1, 1028), f32))
    assert valid.shape == (9, 32) and valid[8].sum() == 1   # K = 1028: the 16-chunk template, one lane in the last chunk
    assert {(K + 127) // 128 <= 6 and 6 or (K + 127) // 128 <= 8 and 8 or 16 for K in LN_KS} == {6, 8, 16}
    assert {K % 128 != 0 for K in LN_KS} == {True, False}


# ---------------------------------------------------------------------------------------------------- 3xFP16 bias columns
def _operand_row(x, hi_scale):
    """[x_h hi_scale | x_l | x_h | FP16_BIAS_ONE, 1, 0 x 6] as the fp16 producers write it (bias_one = FP16_BIAS_ONE)."""
    h = x.half()
    l = ((x - h.float()) * 2048.0).half()
    tail = torch.zeros(x.shape[:-1] + (8,), dtype=torch.float16)
    tail[..., 0], tail[..., 1] = FP16_BIAS_ONE, 1.0
    return torch.cat([(h.float() * hi_scale).half(), l, h, tail], -1)


def _check_bias_columns(x, w, b):
    w16, hi_scale = _w16(w, b)
    assert w16.shape == (w.shape[0], 3 * w.shape[1] + 8) and bool(torch.isfinite(w16.float()).all())
    got = _operand_row(x, hi_scale).double() @ w16.double().t()
    want = FP16_OUT_SCALE * (x.double() @ w.double().t() + b.double())
    mag = FP16_OUT_SCALE * (x.double().abs() @ w.double().abs().t() + b.double().abs())
    assert ((got - want).abs() <= 2.0 ** -21 * mag).all(), ((got - want).abs() / mag).max()
    return hi_scale


@pytest.mark.parametrize("bias_kind", ["randn", "near_guard", "tiny", "zero"])
@pytest.mark.parametrize("wmax", [None, 100.0])
def test_bias_columns_add_the_bias(bias_kind, wmax):
    """x [h 2^a | l | h | 64, 1, 0..] . _w16(W, b) = 2^11 (x W^T + b) to 2^-21 relative, in float64: a = 0 for realistic
    weights, a = 2 with a weight of 100."""
    g = torch.Generator().manual_seed(7)
    x, w = torch.randn(64, 256, generator=g) * 3, torch.randn(48, 256, generator=g) * 0.02
    if wmax is not None:
        w[5, 9] = wmax
    b = {"randn": torch.randn(48, generator=g),
         "near_guard": torch.linspace(-2000.0, 2000.0, 48),
         "tiny": torch.randn(48, generator=g) * 1e-8,
         "zero": torch.zeros(48)}[bias_kind]
    assert _check_bias_columns(x, w, b) == (1.0 if wmax is None else 4.0)


def test_bias_guard():
    """The first bias column holds b_h 2^11 / FP16_BIAS_ONE in fp16: |b| up to 65000 / 32 = 2031.25 passes, beyond raises."""
    w = torch.randn(4, 16) * 0.02
    _check_bias_columns(torch.randn(3, 16), w, torch.tensor([2031.25, -2031.25, 1.0, 0.0]))
    with pytest.raises(OverflowError):
        _w16(w, torch.tensor([0.0, 2031.5, 0.0, 0.0]))
    with pytest.raises(OverflowError):
        _w16(w, torch.tensor([0.0, 0.0, -4000.0, 0.0]))
