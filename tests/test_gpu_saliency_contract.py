"""The kernels that decide which patches and class maps the pipeline produces, at production sizes and at their edges:
pnp_xattn_softmax_fwd and pnp_xattn_softmax_bwd_gradcam (csrc/xattn.cu), pnp_token_merge and pnp_salience_dropout_round
(csrc/gradcam.cu).

References: the oracle (oracle/hotpath.py), an fp64 evaluation of the same formula, or the numpy restatements of
test_saliency_algorithm.py.  Where the kernel follows the reference's fp32 operation order the comparison is bit for bit, and
NaN positions must match exactly.  The xattn kernels keep one row per warp and stride over rows: at most 148 x 8 CTAs of 8 warps
(9472 rows) are resident, so shapes past that run the grid-stride loop.  The row template switches from 16 to 36 items per lane
between K = 512 and 513; K = 1152 is the largest row accepted."""
import numpy as np
import pytest
import torch

from oracle import hotpath as O
from test_saliency_algorithm import PPS, SAVE_LENS, segment_tables, token_merge_restated, wordpiece_tokens

pytestmark = pytest.mark.gpu

RESIDENT_ROWS = 148 * 8 * 8
Q = 2.0 ** -12      # DropOut maps are small multiples of Q: every fp32 sum of them is exact, in any order


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ops():
    from pnp_ovss_b200 import ops as _ops
    return _ops


def _close(got, want, rtol, atol):
    """|got - want| <= atol + rtol |want| elementwise, on whatever device the tensors are; NaN positions must match."""
    got, want = got.double(), want.to(got.device).double()
    assert got.shape == want.shape
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(got), nan)
    err = ((got - want).abs() - (atol + rtol * want.abs()))[~nan]
    assert err.numel() == 0 or err.max().item() <= 0, "max violation %g" % err.max().item()


def _same(a, b):
    """Bit-equal up to the NaN payload."""
    return np.array_equal(a.cpu().numpy(), b.cpu().numpy(), equal_nan=True)


def _same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


# ------------------------------------------------------------------------------------------------ (a) softmax forward
def _softmax_ref(scores, key_mask, scale):
    """fp64 softmax of the kernel's fp32 logits round(round(scores*scale) + key_mask)."""
    x = scores * scale
    if key_mask is not None:
        x = x + key_mask[:, None, None, :]
    return torch.softmax(x.double(), -1)


@pytest.mark.parametrize("K", [1, 2, 31, 32, 33, 442, 512, 513, 577, 785, 1025, 1152])
def test_softmax_fwd_row_lengths(dev, ops, K):
    g = torch.Generator().manual_seed(K)
    s = (torch.randn(3, 12, 7, K, generator=g) * 8).to(dev)
    mask = (torch.rand(3, K, generator=g) * -6).to(dev)
    mask[1, ::3] = -10000.0
    for m in (None, mask):
        _close(ops.softmax_fwd(s, m, 0.125), _softmax_ref(s, m, 0.125), 1e-5, 1e-12)


def test_softmax_fwd_refuses_rows_past_1152(dev, ops):
    from pnp_ovss_b200._lib import PnpError
    with pytest.raises(PnpError):
        ops.softmax_fwd(torch.zeros(1, 1, 1, 1153, device=dev))


def test_softmax_fwd_rows_beyond_one_wave(dev, ops):
    """B=35, 12 heads, T=200 (84000 rows, 9x the resident warps) with a different key mask per image: -10000 on every key but
    one, -10000 mixed with finite values, or finite values only.  In place equals out of place, and two calls are equal."""
    B, h, T, K = 35, 12, 200, 442
    assert B * h * T > 8 * RESIDENT_ROWS
    g = torch.Generator(device=dev).manual_seed(1)
    s = torch.randn(B, h, T, K, device=dev, generator=g) * 8
    mask = torch.rand(B, K, device=dev, generator=g) * -8
    for b in range(0, B, 3):
        mask[b] = -10000.0
        mask[b, (37 * b) % K] = 0.0
    for b in range(1, B, 3):
        mask[b, torch.randperm(K, device=dev, generator=g)[:K // 2]] = -10000.0
    out = ops.softmax_fwd(s, mask, 0.125)
    _close(out, _softmax_ref(s, mask, 0.125), 1e-5, 1e-12)
    for b in range(0, B, 3):
        assert torch.equal(out[b, :, :, (37 * b) % K], torch.ones(h, T, device=dev))
    assert _same_bits(ops.softmax_fwd(s, mask, 0.125), out)
    s_in = s.clone()
    assert ops.softmax_fwd(s_in, mask, 0.125, out=s_in).data_ptr() == s_in.data_ptr()
    assert _same_bits(s_in, out)


@pytest.mark.parametrize("K", [442, 1025])
def test_softmax_fwd_nan_and_inf_rows(dev, ops, K):
    """A row holding NaN, a row holding +inf and a row of -inf give NaN where torch's softmax does; the other rows are unharmed."""
    g = torch.Generator().manual_seed(K)
    s = torch.randn(2, 12, 5, K, generator=g) * 8
    s[0, 0, 0, 5] = float("nan")
    s[0, 1, 2, K - 1] = float("inf")
    s[1, 3, 4, :] = float("-inf")
    s[1, 5, 1, :K // 2] = float("-inf")
    got = ops.softmax_fwd(s.to(dev), None, 0.125).cpu()
    want = torch.softmax(s * 0.125, -1)
    assert torch.equal(torch.isnan(got), torch.isnan(want))
    assert torch.isnan(got).any(-1).sum() == 3
    _close(got, _softmax_ref(s, None, 0.125), 1e-5, 1e-12)


# ------------------------------------------------------------------------------------------------ (a) backward + GradCAM
def _gradcam_ref(probs, dprobs, token_mask, head):
    """BITM:427-433 as oracle.gradcam_from_capture writes it, for any K (the oracle needs K-1 = P*P)."""
    T = probs.shape[2]
    m = token_mask[:, None, :T, None]
    g = probs[:, :, :, 1:] * dprobs[:, :, :, 1:].clamp(0) * m
    g[g < 0] = 0
    return g[:, head, 1:]


def _gradcam_oracle(probs, dprobs, token_mask, head):
    K = probs.shape[3]
    want = _gradcam_ref(probs, dprobs, token_mask, head)
    P = int(round((K - 1) ** 0.5))
    if P * P == K - 1:
        o = O.gradcam_head(probs, dprobs, token_mask, P, head)
        assert _same(o.reshape(want.shape), want)
    return want


def _dscores_ref(probs, dprobs, scale):
    p, d = probs.double(), dprobs.double()
    return p * (d - (p * d).sum(-1, keepdim=True)) * scale


def _inputs(B, h, T, K, seed, device="cpu"):
    g = torch.Generator(device=device).manual_seed(seed)
    probs = torch.softmax(torch.randn(B, h, T, K, device=device, generator=g) * 3, -1)
    dprobs = torch.randn(B, h, T, K, device=device, generator=g) * 1e-3
    token_mask = (torch.rand(B, 500, device=device, generator=g) < 0.6).long()    # arbitrary 0/1 pattern, not a prefix
    return probs, dprobs, token_mask


def _check_bwd(ops, probs, dprobs, token_mask, head, scale=0.125):
    want = _gradcam_oracle(probs, dprobs, token_mask, head)
    ds, cam = ops.softmax_bwd_gradcam(probs, dprobs, token_mask, head, scale, True, True)
    assert _same(cam, want)
    ref = _dscores_ref(probs, dprobs, scale)
    _close(ds, ref, 1e-4, 1e-5 * ref.nan_to_num(0.0).abs().max().item())
    ds2, cam2 = ops.softmax_bwd_gradcam(probs, dprobs, token_mask, head, scale, False, True)
    assert ds2 is None and _same_bits(cam2, cam)
    return ds, cam


@pytest.mark.parametrize("K", [2, 33, 512, 513, 577, 785, 1025, 1152])
@pytest.mark.parametrize("T", [1, 2, 9])
@pytest.mark.parametrize("head", [0, 11])
def test_softmax_bwd_gradcam_shapes(dev, ops, K, T, head):
    probs, dprobs, token_mask = _inputs(3, 12, T, K, 31 * K + 7 * T + head)
    _check_bwd(ops, probs.to(dev), dprobs.to(dev), token_mask.to(dev), head)


def test_softmax_bwd_gradcam_with_nothing_to_write(dev, ops):
    """B = 0, or frozen mode with T = 1 (no GradCAM rows): empty outputs of the right shapes, and a bad head still refused."""
    from pnp_ovss_b200._lib import PnpError
    for B, T, need_ds in ((0, 9, True), (0, 9, False), (3, 1, False)):
        probs, dprobs, token_mask = _inputs(B, 12, T, 442, 1, device=dev)
        ds, cam = ops.softmax_bwd_gradcam(probs, dprobs, token_mask, 9, 0.125, need_ds, True)
        assert cam.shape == (B, T - 1, 441) and (ds is None) != need_ds and (ds is None or ds.shape == probs.shape)
        with pytest.raises(PnpError):
            ops.softmax_bwd_gradcam(probs, dprobs, token_mask, 12, 0.125, need_ds, True)


@pytest.mark.parametrize("B,T", [(35, 30), (35, 300)])
def test_softmax_bwd_gradcam_rows_beyond_one_wave(dev, ops, B, T):
    """Past the resident warps in full mode (35x12x30 = 12600 rows) and in frozen mode (B=35, T=300: 10465 GradCAM rows)."""
    assert B * 12 * T > RESIDENT_ROWS and (T < 100 or B * (T - 1) > RESIDENT_ROWS)
    probs, dprobs, token_mask = _inputs(B, 12, T, 442, T, device=dev)
    _check_bwd(ops, probs, dprobs, token_mask, 9)


@pytest.mark.parametrize("K", [442, 1025])
def test_softmax_bwd_dscores_may_alias_dprobs(dev, ops, K):
    from pnp_ovss_b200 import _lib
    B, h, T = 35, 12, 30
    probs, dprobs, token_mask = _inputs(B, h, T, K, K, device=dev)
    ds, cam = ops.softmax_bwd_gradcam(probs, dprobs, token_mask, 9, 0.125, True, True)
    buf = dprobs.clone()
    cam2 = torch.empty_like(cam)
    ops.check(_lib.load().pnp_xattn_softmax_bwd_gradcam(ops._p(probs), ops._p(buf), ops._p(buf), ops._p(token_mask), 500,
                                                        ops._p(cam2), B, h, T, K, 0.125, 9, ops._stream()), "in place")
    assert _same_bits(buf, ds) and _same_bits(cam2, cam)


@pytest.mark.parametrize("K", [442, 1025])
def test_gradcam_nan_in_dprobs_propagates(dev, ops, K):
    """torch's clamp(0) keeps a NaN gradient NaN, so the reference's GradCAM is NaN there (unless the token mask is 0 -- NaN * 0
    is still NaN)."""
    probs, dprobs, token_mask = _inputs(4, 12, 9, K, K)
    dprobs[0, 9, 3, 10] = float("nan")
    dprobs[1, 9, 1, 1:40] = float("nan")
    dprobs[2, 9, 5, K - 1] = float("nan")
    dprobs[3, 4, 2, 7] = float("nan")      # another head: dscores only
    token_mask[1, 1] = 0
    ds, cam = _check_bwd(ops, probs.to(dev), dprobs.to(dev), token_mask.to(dev), 9)
    assert int(torch.isnan(cam).sum()) == 1 + 39 + 1


@pytest.mark.parametrize("K", [442, 1025])
def test_gradcam_nan_in_probs_propagates(dev, ops, K):
    probs, dprobs, token_mask = _inputs(4, 12, 9, K, K + 1)
    probs[0, 9, 3, 10] = float("nan")
    probs[1, 9, 2, 1:40] = float("nan")
    dprobs[1, 9, 2, 1:20] = -1.0            # NaN * 0 is NaN too
    ds, cam = _check_bwd(ops, probs.to(dev), dprobs.to(dev), token_mask.to(dev), 9)
    assert int(torch.isnan(cam).sum()) == 1 + 39


# ------------------------------------------------------------------------------------------------ (b) token merge
def _merge_both_ways(dev, ops, g, start, length, div, poison=False):
    """pnp_token_merge, bit-equal to the restatement.  poison: the output block held NaN before the call."""
    args = [torch.from_numpy(a).to(dev) for a in (g, start, length, div)]
    if poison:
        junk = torch.full((g.shape[0], start.shape[1], g.shape[2]), float("nan"), device=dev)
        ptr = junk.data_ptr()
        del junk
    got = ops.token_merge(*args, 3, int((start + length).max()))
    assert not poison or got.data_ptr() == ptr      # the merge wrote into the NaN-filled block
    assert np.array_equal(got.cpu().numpy(), token_merge_restated(g, start, length, div, 3), equal_nan=True)
    return got


@pytest.mark.parametrize("C", [1, 20, 150, 171])
@pytest.mark.parametrize("PP", PPS)
def test_token_merge_random_segment_tables(dev, ops, C, PP):
    """Random tables: seg_len 0..6, div 1 or the word length; the output block was NaN before the call, so seg_len = 0 must
    write zeros rather than leave the block as it was."""
    B, rows = 35, 200
    rng = np.random.default_rng(C * PP)
    start = rng.integers(0, rows, (B, C)).astype(np.int32)
    length = rng.integers(0, 7, (B, C)).astype(np.int32)
    length[0, 0] = 0
    div = np.where(rng.random((B, C)) < 0.5, np.maximum(length, 1), 1).astype(np.float32)
    g = (rng.standard_normal((B, 3 + rows + 7, PP)) * 4).astype(np.float32)
    got = _merge_both_ways(dev, ops, g, start, length, div, poison=True)
    zero = torch.from_numpy(length == 0).to(dev)
    assert (got[zero].view(torch.int32) == 0).all()


@pytest.mark.parametrize("C", [1, 20, 150, 171])
@pytest.mark.parametrize("PP", [441, 1024])
def test_token_merge_wordpiece_captions(dev, ops, C, PP):
    """Tables from host.build_token_segments on random WordPiece captions of C words (up to 6 pieces each; every fourth caption
    unsplit, where the reference takes the rows as they are): bit-equal to the oracle's reference loop."""
    B = 35
    rng = np.random.default_rng(C + PP)
    captions = []
    for b in range(B):
        pieces = [1] * C if b % 4 == 0 else rng.integers(1, 7, C).tolist()
        captions.append((wordpiece_tokens(pieces), C))
    Tm = 3 + max(len(t) for t, _ in captions) + 1
    g = (rng.standard_normal((B, Tm, PP)) * 4).astype(np.float32)
    start, length, div = segment_tables(captions)
    got = _merge_both_ways(dev, ops, g, start, length, div).cpu().numpy()
    P = int(round(PP ** 0.5))
    for b, (toks, n) in enumerate(captions):
        rows = torch.from_numpy(g[b, :3 + len(toks) + 1]).reshape(-1, P, P)
        want = O.mean_over_filtered_label_tokens(toks, rows, n).numpy()
        assert np.array_equal(got[b].reshape(want.shape), want), b


# ------------------------------------------------------------------------------------------------ (c) Salience DropOut round
def _dropout_round_ref(g, agg, chosen, n_prev, imgs, norm_imgs, P, patch, save_len, r):
    """One round of oracle.salience_dropout (DRV:589-647, 716-721) with argsort kind="stable".  g [B,Tm,P,P] on the CPU; chosen
    numpy [B, stride] (updated); imgs / norm_imgs on the device.  Returns (pred, agg, imgs, norm_imgs)."""
    B = g.shape[0]
    pred = g.clone()
    for b in range(B):
        for idx in chosen[b, :n_prev]:
            pred[b][:, idx // P, idx % P] = 0
    agg = pred + pred if r == 0 else agg + pred
    for b in range(B):
        sort_union = g[b][3:-1, :, :].sum(dim=0).flatten().numpy().copy()
        for idx in chosen[b, :n_prev]:
            sort_union[idx] = 0
        chosen[b, n_prev:n_prev + save_len] = np.argsort(sort_union, kind="stable")[-save_len:]
    cells = np.zeros((B, P * P), bool)
    np.put_along_axis(cells, chosen[:, n_prev:n_prev + save_len].astype(np.int64), True, 1)
    pix = torch.from_numpy(cells.reshape(B, P, P)).to(imgs.device if imgs is not None else "cpu")
    pix = pix.repeat_interleave(patch, 1).repeat_interleave(patch, 2)
    if imgs is not None:
        imgs = imgs.masked_fill(pix[:, None], 0.0)
    if norm_imgs is not None:
        norm_imgs = norm_imgs.masked_fill(pix[..., None], 0.0)
    return pred, agg, imgs, norm_imgs


def _maps(rng, B, Tm, P, save_len, kinds=5):
    """Per image: 0 small random integers; 1 an all-zero map; 2 2*save_len+3 cells tied at the top score, so that the ties
    straddle the top-k boundary in the third round; 3 negative and positive integers; 4 integers with +inf and -inf cells.
    All in units of Q.  The map is the same every round, so previously chosen cells would win again if they were not dropped."""
    PP = P * P
    g = rng.integers(0, 8, (B, Tm, PP)).astype(np.float32)
    for b in range(B):
        kind = b % kinds
        if kind == 1:
            g[b] = 0
        elif kind == 2:
            g[b] = rng.integers(0, 3, (Tm, PP))
            g[b][3:Tm - 1, rng.choice(PP, 2 * save_len + 3, replace=False)] = 3
        elif kind == 3:
            g[b] = rng.integers(-6, 6, (Tm, PP))
        elif kind == 4:
            cells = rng.choice(PP, 10, replace=False)
            g[b, 3, cells[:4]] = np.inf
            g[b, 3, cells[4:]] = -np.inf
    return g * np.float32(Q)


def _run_rounds(dev, ops, maps, P, patch, save_len, R, imgs=None, norm_imgs=None):
    """Calls the kernel round by round as pipeline.salience_dropout_loop does and compares every output with the reference."""
    B, Tm = maps.shape[:2]
    S = P * patch
    if imgs is None:
        gen = torch.Generator(device=dev).manual_seed(P * patch + save_len)
        imgs = torch.randn(B, 3, S, S, device=dev, generator=gen)
        norm_imgs = torch.randn(B, S, S, 3, device=dev, generator=gen)
    chosen = torch.full((B, save_len * R), -1, dtype=torch.int32, device=dev)
    chosen_ref = np.full((B, save_len * R), -1, np.int64)
    agg = torch.empty(B, Tm, P, P, device=dev)
    ens = torch.empty_like(agg)
    agg_ref, imgs_ref, norm_ref = None, imgs.clone(), norm_imgs.clone()
    g = torch.from_numpy(maps).reshape(B, Tm, P, P)
    for r in range(R):
        ops.salience_dropout_round(g.to(dev), agg, chosen, save_len * r, imgs, norm_imgs, P, patch, 3, Tm - 1, save_len, r,
                                   ensemble_r=ens)
        pred, agg_ref, imgs_ref, norm_ref = _dropout_round_ref(g, agg_ref, chosen_ref, save_len * r, imgs_ref, norm_ref, P, patch,
                                                               save_len, r)
        assert np.array_equal(chosen.cpu().numpy(), chosen_ref), r
        assert _same(ens, pred) and _same(agg, agg_ref), r
        assert torch.equal(imgs, imgs_ref) and torch.equal(norm_imgs, norm_ref), r
    return chosen, agg, imgs, norm_imgs


@pytest.mark.parametrize("P", [21, 24, 28, 32])
@pytest.mark.parametrize("save_len", SAVE_LENS)
@pytest.mark.parametrize("patch", [16, 8])
def test_dropout_rounds_match_the_reference_sequence(dev, ops, P, save_len, patch):
    """B=35, 4 rounds: the chosen cells in the reference's order (ascending score, ties by index), agg, ensemble_r and the whole
    imgs / norm_imgs tensors (exactly the new blocks zeroed) bit-equal to the reference."""
    maps = _maps(np.random.default_rng(P * save_len + patch), 35, 9, P, save_len)
    _run_rounds(dev, ops, maps, P, patch, save_len, 4)


@pytest.mark.parametrize("P", [21, 32])
def test_dropout_empty_class_row_range(dev, ops, P):
    """Tm = 4: the score rows [3, Tm-1) are empty, every score is 0 and the largest indices win (previously chosen ones too)."""
    maps = _maps(np.random.default_rng(P), 35, 4, P, 10)
    chosen, _, _, _ = _run_rounds(dev, ops, maps, P, 16, 10, 4)
    assert (chosen[:, :10].cpu().numpy() == np.arange(P * P - 10, P * P)).all()


def test_dropout_optional_outputs(dev, ops):
    """imgs=None, norm_imgs=None or agg=None leave every other output as the full call writes it."""
    B, Tm, P, patch, save_len = 35, 9, 24, 16, 10
    S = P * patch
    g = torch.from_numpy(_maps(np.random.default_rng(5), B, Tm, P, save_len)).reshape(B, Tm, P, P).to(dev)
    gen = torch.Generator(device=dev).manual_seed(5)
    imgs0 = torch.randn(B, 3, S, S, device=dev, generator=gen)
    norm0 = torch.randn(B, S, S, 3, device=dev, generator=gen)
    prev = torch.randint(0, P * P, (B, 2 * save_len), device=dev, generator=gen, dtype=torch.int32)
    agg0 = torch.randn(B, Tm, P, P, device=dev, generator=gen)

    def run(with_imgs, with_norm, with_agg):
        chosen = torch.cat([prev, torch.full((B, save_len), -1, dtype=torch.int32, device=dev)], 1)
        imgs, norm, agg = imgs0.clone(), norm0.clone(), agg0.clone()
        ens = torch.empty_like(agg)
        ops.salience_dropout_round(g, agg if with_agg else None, chosen, 2 * save_len, imgs if with_imgs else None,
                                   norm if with_norm else None, P, patch, 3, Tm - 1, save_len, 2, ensemble_r=ens)
        return chosen, imgs, norm, agg, ens

    full = run(True, True, True)
    assert not torch.equal(full[1], imgs0) and not torch.equal(full[2], norm0) and not _same(full[3], agg0)
    for flags in ((False, True, True), (True, False, True), (True, True, False)):
        part = run(*flags)
        want = list(full)
        want[1] = want[1] if flags[0] else imgs0
        want[2] = want[2] if flags[1] else norm0
        want[3] = want[3] if flags[2] else agg0
        for a, b in zip(part, want):
            assert _same(a, b), flags


def _nan_maps(rng, B, Tm, P, n_finite=None):
    """Small integer maps (units of Q) with NaN in the score rows: a few NaN cells per image, or NaN everywhere but n_finite cells."""
    PP = P * P
    g = rng.integers(-4, 8, (B, Tm, PP)).astype(np.float32)
    for b in range(B):
        if n_finite is None:
            cells = rng.choice(PP, 3 + b % 5, replace=False)
            g[b, 3 + b % (Tm - 4), cells] = np.nan
        else:
            keep = rng.choice(PP, n_finite, replace=False)
            nan = np.ones(PP, bool)
            nan[keep] = False
            g[b, 3, nan] = np.nan
        g[b, 0, rng.choice(PP, 2, replace=False)] = np.nan       # outside the score rows: agg / ensemble_r only
    return g * np.float32(Q)


@pytest.mark.parametrize("P", [21, 32])
@pytest.mark.parametrize("save_len", SAVE_LENS)
def test_dropout_nan_scores_are_chosen_first(dev, ops, P, save_len):
    """np.argsort sorts NaN last, so the reference drops NaN-scored cells first.  Three runs give the same cells."""
    maps = _nan_maps(np.random.default_rng(P + save_len), 35, 9, P)
    runs = [_run_rounds(dev, ops, maps, P, 16, save_len, 4)[0] for _ in range(3)]
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])


@pytest.mark.parametrize("P", [21, 32])
@pytest.mark.parametrize("save_len", SAVE_LENS)
def test_dropout_mostly_nan_scores(dev, ops, P, save_len):
    """Every score NaN but four: the reference's order, and only blocks of valid cells are written.  imgs and norm_imgs sit
    inside larger buffers whose margins must stay as they were."""
    B, Tm, patch = 35, 9, 16
    S = P * patch
    maps = _nan_maps(np.random.default_rng(P * save_len), B, Tm, P, n_finite=4)
    n, margin = B * 3 * S * S, 1 << 20
    gen = torch.Generator(device=dev).manual_seed(P)
    bufs = [torch.randn(n + 2 * margin, device=dev, generator=gen) for _ in range(2)]
    before = [b.clone() for b in bufs]
    imgs = bufs[0][margin:margin + n].view(B, 3, S, S)
    norm = bufs[1][margin:margin + n].view(B, S, S, 3)
    chosen, _, _, _ = _run_rounds(dev, ops, maps, P, patch, save_len, 4, imgs, norm)
    c = chosen.cpu().numpy()
    assert c.min() >= 0 and c.max() < P * P
    for b, b0 in zip(bufs, before):
        assert torch.equal(b[:margin], b0[:margin]) and torch.equal(b[margin + n:], b0[margin + n:])
