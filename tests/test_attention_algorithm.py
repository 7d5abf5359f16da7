"""CPU restatement of the arithmetic contract of the tcgen05 attention kernel (pnp_ovss_b200/csrc/attention.cu), in numpy:
  * every fp32 operand x is split exactly into x = h + l 2^-11 (h = fp16(x), l = fp16((x - h) 2^11)) and a product a.b is evaluated as
    a_h b_h + 2^-11 (a_l b_h + a_h b_l) with fp32 accumulation (the dropped a_l b_l term is ~2^-22 relative);
  * keys stream in tiles of 64; a row's softmax subtracts a reference m_used that is refreshed -- and O, l rescaled -- only when the
    row maximum (rounded UP to bf16, the bound both threads of a row exchange) has outgrown it by more than 2^8 in the exp2 domain.
Any common shift is exact for a softmax, so the result must equal the plain fp64 attention to fp32 grade; p stays below 2^8 (1 + 2^-7).
These are the properties the -m gpu tests rely on when they compare the kernel with an fp64 evaluation.  The bound is exact only while
|m_used| < 2^11 (a bf16 ulp of at most 8, so the largest p of a row stays >= 2^-8, in fp16's normal range); beyond it the kernel raises
its overflow flag, restated here as expected_overflow_flag (tests/test_gpu_attention_contract.py compares the kernel's flag with it)."""
import numpy as np
import pytest


def split_hi_lo(x):
    x = np.asarray(x, np.float32)
    h = x.astype(np.float16)
    l = ((x - h.astype(np.float32)) * np.float32(2048.0)).astype(np.float16)
    return h, l


def product_3x(a, b):
    """a [M,K] . b [N,K]^T with the three fp16 products accumulated in fp32 (main and correction accumulators apart)."""
    ah, al = split_hi_lo(a)
    bh, bl = split_hi_lo(b)
    f = lambda t: t.astype(np.float32)
    main = f(ah) @ f(bh).T
    corr = f(al) @ f(bh).T + f(ah) @ f(bl).T
    return main + corr * np.float32(1.0 / 2048.0)


def bf16_round_up(x):
    u = np.asarray(x, np.float32).view(np.uint32).copy()
    neg = (u & 0x80000000) != 0
    u = np.where(neg, u & 0xFFFF0000, (u + 0xFFFF) & 0xFFFF0000).astype(np.uint32)
    return u.view(np.float32)


FP16_MAX = 65504.0
BOUND_LIMIT = 2048.0        # |m_used| (exp2 domain, ~1420 in natural logits) from which the kernel raises its overflow flag


def attention_tiled(q, k, v, scale, tile=64, threshold=8.0):
    """One head: q [Lq,D], k, v [L,D] -> (o [Lq,D], largest p seen, number of rescales, final bound m_used [Lq])."""
    L = k.shape[0]
    qs = (q * np.float32(scale * 1.4426950408889634)).astype(np.float32)
    m_used = np.full(q.shape[0], -np.inf, np.float32)
    l = np.zeros(q.shape[0], np.float32)
    o = np.zeros((q.shape[0], v.shape[1]), np.float32)
    p_max, rescales = 0.0, 0
    for k0 in range(0, L, tile):
        s = product_3x(qs, k[k0:k0 + tile])                         # exp2-domain scores of the tile
        mx = bf16_round_up(s.max(1))
        grow = mx > m_used + np.float32(threshold)                  # always on the first tile
        with np.errstate(over="ignore"):                              # rows that do not grow may overflow here; the value is discarded
            alpha = np.where(grow, np.exp2(m_used - mx), np.float32(1.0)).astype(np.float32)
        if k0 > 0:
            rescales += int(grow.sum())
            o *= alpha[:, None]
            l *= alpha
        m_used = np.where(grow, mx, m_used)
        p = np.exp2(s - m_used[:, None]).astype(np.float32)
        p_max = max(p_max, float(p.max()))
        l += p.sum(1)
        o += product_3x(p, v[k0:k0 + tile].T)                       # P V as a product against V^T rows
    return o / l[:, None], p_max, rescales, m_used


def expected_overflow_flag(q, k, v, scale, in_scale=1.0):
    """The overflow flag of pnp_attention_fp16x3 for one head in `out` mode (q, k, v as stored, each value times 1/in_scale): a k or v
    value times in_scale, or a q value times in_scale * scale * log2(e), outside fp16's range or NaN; or a row whose final bound
    m_used is not below 2^11 in magnitude."""
    f = lambda x, s: not (np.abs(np.asarray(x, np.float64) * s) <= FP16_MAX).all()
    if f(q, in_scale * scale * 1.4426950408889634) or f(k, in_scale) or f(v, in_scale):
        return True
    x = lambda t: (np.asarray(t, np.float32) * np.float32(in_scale)).astype(np.float32)
    with np.errstate(all="ignore"):
        m_used = attention_tiled(x(q), x(k), x(v), scale)[3]
    return not (np.abs(m_used) < BOUND_LIMIT).all()


def shifted_head(c, L=442, seed=0, scale=0.125):
    """q, k, v of one head whose scores are randn-like plus exactly c (natural units) in every row: k[:, 0] = 1, q[:, 0] = c / scale."""
    rng = np.random.default_rng(seed)
    q = rng.standard_normal((L, 64)).astype(np.float32)
    k = rng.standard_normal((L, 64)).astype(np.float32)
    v = rng.standard_normal((L, 64)).astype(np.float32)
    q[:, 0] = np.float32(c / scale)
    k[:, 0] = 1.0
    return q, k, v


@pytest.mark.parametrize("L,spread", [(442, 1.0), (130, 6.0), (64, 0.2), (37, 3.0)])
def test_tiled_lazy_rescale_softmax_equals_plain_attention(L, spread):
    rng = np.random.default_rng(L)
    q = (rng.standard_normal((96, 64)) * spread).astype(np.float32)
    k = (rng.standard_normal((L, 64)) * spread).astype(np.float32)
    v = rng.standard_normal((L, 64)).astype(np.float32)
    scale = 0.125
    s = (q.astype(np.float64) @ k.astype(np.float64).T) * scale
    w = np.exp(s - s.max(1, keepdims=True))
    truth = (w / w.sum(1, keepdims=True)) @ v.astype(np.float64)
    got, p_max, rescales, _ = attention_tiled(q, k, v, scale)
    err = np.abs(got - truth).max() / np.abs(truth).max()
    assert err < (3e-6 if spread <= 3.0 else 1e-5), err               # fp32 grade (plain fp16 operands: ~1e-3); scores of +-700 at spread 6
    assert p_max <= 256.0 * (1 + 2.0 ** -7)                           # the bound the fp16 pairs rely on
    plain16 = (w / w.sum(1, keepdims=True)).astype(np.float16).astype(np.float64) @ v.astype(np.float16).astype(np.float64)
    assert np.abs(plain16 - truth).max() / np.abs(truth).max() > 30 * err
    if spread >= 3.0 and L > 64:
        assert rescales > 0                                           # the lazy path is exercised, not just tile 0


def test_split_is_exact_and_three_products_recover_fp32_products():
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(4096) * 10.0 ** rng.uniform(-3, 3, 4096)).astype(np.float32)
    h, l = split_hi_lo(x)
    back = h.astype(np.float64) + l.astype(np.float64) / 2048.0
    assert np.abs(back - x.astype(np.float64)).max() <= np.abs(x).max() * 2.0 ** -21   # 22-23 significant bits survive the pair
    a = rng.standard_normal((32, 64)).astype(np.float32)
    b = rng.standard_normal((48, 64)).astype(np.float32)
    truth = a.astype(np.float64) @ b.astype(np.float64).T
    e3 = np.abs(product_3x(a, b) - truth).max()
    e16 = np.abs(a.astype(np.float16).astype(np.float64) @ b.astype(np.float16).astype(np.float64).T - truth).max()
    e32 = np.abs((a @ b.T).astype(np.float64) - truth).max()
    assert e3 <= 8 * e32 + 1e-6 and e3 * 100 < e16


def _attention_fp32(q, k, v, scale):
    s = (q @ k.T) * np.float32(scale)
    w = np.exp(s - s.max(1, keepdims=True))
    return (w / w.sum(1, keepdims=True)) @ v


def _attention_fp64(q, k, v, scale):
    return _attention_fp32(*(t.astype(np.float64) for t in (q, k, v)), scale)


SHIFTS_IN_RANGE = (-1400, -300, 0, 50, 300, 1000, 1400)
SHIFTS_PAST_BOUND = (-6000, 6000, 12000, 30000)


def test_common_shift_sweep_is_fp32_grade_below_the_bound_and_flagged_past_it():
    """A common shift c of every score leaves a softmax unchanged.  While the final bound stays below 2^11 (exp2 domain) the restatement
    is fp32-grade at every c; past it the bf16 bound loses the row's largest p (output ~0 or NaN) -- the case the flag reports."""
    scale = 0.125
    lost = 0
    for c in SHIFTS_IN_RANGE + SHIFTS_PAST_BOUND:
        q, k, v = shifted_head(c, L=200, seed=3)
        truth = _attention_fp64(q, k, v, scale)
        sc = np.abs(truth).max()
        e32 = np.abs(_attention_fp32(q, k, v, scale) - truth).max() / sc
        with np.errstate(all="ignore"):
            got, _, _, m_used = attention_tiled(q, k, v, scale)
        e_got = np.abs(got - truth).max() / sc
        flagged = expected_overflow_flag(q, k, v, scale)
        assert flagged == (abs(c) >= 6000), (c, np.abs(m_used).max())
        if not flagged:
            assert np.abs(m_used).max() < BOUND_LIMIT
            assert e_got <= 4 * e32 + 4e-6, (c, e_got, e32)
        elif not e_got <= 1e-2:                                           # NaN counts as lost
            lost += 1
    assert lost >= 1                                                      # why the flag threshold exists


def test_expected_overflow_flag_names_each_operand():
    q, k, v = shifted_head(0, L=70, seed=4)
    assert not expected_overflow_flag(q, k, v, 0.125)
    for which, val in ((0, 4e5), (1, 7e4), (2, 7e4), (0, np.nan), (1, np.nan)):
        t = [q.copy(), k.copy(), v.copy()]
        t[which][5, 9] = val
        assert expected_overflow_flag(*t, 0.125), (which, val)
    assert not expected_overflow_flag(q * 4096, k * 4096, v * 4096, 0.125, in_scale=1.0 / 4096)
