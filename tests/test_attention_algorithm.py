"""CPU restatement of the arithmetic contract of the tcgen05 attention kernel (pnp_ovss_b200/csrc/attention.cu), in numpy:
  * every fp32 operand x is split exactly into x = h + l 2^-11 (h = fp16(x), l = fp16((x - h) 2^11)) and a product a.b is evaluated as
    a_h b_h + 2^-11 (a_l b_h + a_h b_l) with fp32 accumulation (the dropped a_l b_l term is ~2^-22 relative);
  * keys stream in tiles of 64; a row's softmax subtracts a reference m_used that is refreshed -- and O, l rescaled -- only when the
    row maximum (rounded UP to bf16, the bound both threads of a row exchange) has outgrown it by more than 2^8 in the exp2 domain.
Any common shift is exact for a softmax, so the result must equal the plain fp64 attention to fp32 grade; p stays below 2^8 (1 + 2^-7).
These are the properties the -m gpu tests rely on when they compare the kernel with an fp64 evaluation."""
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


def attention_tiled(q, k, v, scale, tile=64, threshold=8.0):
    """One head: q [Lq,D], k, v [L,D] -> (o [Lq,D], largest p seen, number of rescales)."""
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
    return o / l[:, None], p_max, rescales


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
    got, p_max, rescales = attention_tiled(q, k, v, scale)
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
