"""The post-processing kernels (pnp_ovss_b200/csrc/upsample_blur.cu, confusion.cu) against plain fp64 references at real
ground-truth shapes and at the edges of their contract: the direct Gaussian blur, threshold + upsample, the fused low-rank
group, argmax and the confusion histogram, their size limits, and non-finite inputs of the raw blur.

Which branch of the host planners each shape reaches is stated and checked in test_postprocess_algorithm.py, together with the
fp64 operators used here: G (reflect-mode Gaussian, scipy's weights) and U (bilinear, align_corners=True).

Bounds.
- Raw blur of a map x against gaussian_filter(float64 x): each pass is one fp32 FMA chain of T = 2 lw + 1 taps with weights
  rounded to fp32, so it is off by at most (T + 1) u sum_j w_j |x| <= (T + 1) u max|x| (u = 2^-24; the chain's T roundings
  plus the weights' one), and two passes by 2 (T + 1) u max|x|.  BLUR_ULP_BOUND below.
- A unit impulse blurs to w_y w_x (each a sum of at most two weights where the reflection folds): at most 8 u relative --
  two weight roundings, at most two additions, one product, with slack -- on every output that is not exactly zero, the far
  tail taps included; every other output is exactly zero.
- Fused low-rank maps within 5e-6 of fp64 after the min/max normalisation, unaries within 3e-5 (the bounds of
  test_gpu_kernels.py, which the fp64 closed form keeps).  Labels are exact wherever the fp64 winner leads by more than
  twice the map bound."""
import functools

import numpy as np
import pytest
import torch

from pnp_ovss_b200 import synthetic as synth
from test_postprocess_algorithm import (ARGMAX_C, BLUR_PLAIN_VS_TMA, BLUR_SCALE, BLUR_SHAPES, CONFUSION_N_CLASS, CONFUSION_SHAPES,
                                        LOWRANK_HUGE_C, LOWRANK_NO_BG_LARGE, LOWRANK_P, LOWRANK_SHAPES, LOWRANK_TINY, LOWRANK_WIDE_C,
                                        blur_plan, gauss_matrix, gauss_weights, interp_matrix)

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
MAP_BOUND, UNARY_BOUND = 5e-6, 3e-5
IMPULSE_REL = 8 * U32
PNP_ERR_INVALID_ARGUMENT = -1
OBSERVED = {}      # largest error seen per comparison, printed with -s


def BLUR_ULP_BOUND(sigma, xmax):
    return 2 * (2 * int(4.0 * sigma + 0.5) + 2) * U32 * xmax


def _observe(key, err, bound):
    OBSERVED[key] = max(OBSERVED.get(key, 0.0), float(err))
    print("%s: max error %.3g (bound %.3g)" % (key, err, bound))


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


@pytest.fixture(scope="module")
def O():
    from oracle import hotpath
    return hotpath


@functools.lru_cache(maxsize=None)
def _G(n, sigma):
    return gauss_matrix(n, sigma)


@functools.lru_cache(maxsize=None)
def _A(n, P, sigma):
    """G U: the upsample-then-blur operator of one axis, [n, P] in float64."""
    return _G(n, sigma) @ interp_matrix(n, P)


def _sigma(H, W):
    return BLUR_SCALE * max(H, W)


def _offset_view(x):
    """The same values in storage offset by one float: contiguous, but only 4-byte aligned."""
    buf = torch.empty(x.numel() + 1, dtype=x.dtype, device=x.device)
    v = buf[1:].view(x.shape)
    v.copy_(x)
    assert v.data_ptr() % 16 == 4
    return v


def _same(got, want):
    """Bit-equal, except that a NaN only has to be a NaN."""
    assert got.shape == want.shape
    assert torch.equal(got.isnan(), want.isnan())
    assert torch.equal(got.nan_to_num(0.0, 7.0, -7.0), want.nan_to_num(0.0, 7.0, -7.0))


def _minmax_is_amin_amax(raw, mm):
    _same(mm[:, 0], raw.flatten(1).amin(1))
    _same(mm[:, 1], raw.flatten(1).amax(1))


# ================================================================================================ A. direct blur
def _blur_maps(H, W):
    rng = np.random.default_rng(H * 7919 + W)
    x = rng.random((2, H, W))
    x[1] = x[1] > 0.7                   # binary, like the background indicator
    return x.astype(np.float32)


@pytest.mark.parametrize("shape", sorted(BLUR_SHAPES))
def test_blur_matches_scipy(dev, ops, shape):
    from scipy.ndimage import gaussian_filter
    H, W = shape
    s = _sigma(H, W)
    x = _blur_maps(H, W)
    raw, mm = ops.gaussian_blur(torch.from_numpy(x).to(dev), s, normalize=False)
    _minmax_is_amin_amax(raw, mm)
    raw = raw.cpu().numpy()
    for i in range(x.shape[0]):
        want = gaussian_filter(x[i].astype(np.float64), s)
        err = np.abs(raw[i] - want).max()
        bound = BLUR_ULP_BOUND(s, 1.0)
        _observe("blur %dx%d map %d" % (H, W, i), err, bound)
        assert err <= bound


def _impulse_sites(H, W):
    """(y, x) impulse positions: on and either side of the V row-tile, V strip, H row-block, H sweep and H column-tile
    boundaries, within lw of every edge (the reflection folds) and in the corners."""
    p = blur_plan(1, H, W, _sigma(H, W))
    lw = p["lw"]

    def around(edges, n):
        out = set()
        for e in edges:
            out.update(v for v in (e - 1, e, e + 1) if 0 <= v < n)
        return out

    v_edges = [k * p["v_rows"] for k in range(1, p["v_tiles"])]
    v_edges = v_edges[:2] + v_edges[-1:]                            # the first two and the last row-tile boundaries
    rows = around(v_edges + [32, (H // 64) * 32], H) | {min(lw - 1, H - 1), max(H - lw, 0), 1, H - 2}
    sweep = p["h_groups"] * 16
    c_edges = [k * p["h_cols"] for k in range(1, p["h_tiles"])][:2] + [sweep] + [p["v_cols"]]
    cols = around(c_edges, W) | {min(lw - 1, W - 1), max(W - lw, 0), 1, W - 2}
    rows, cols = sorted(r for r in rows if 0 <= r < H), sorted(c for c in cols if 0 <= c < W)
    n = max(len(rows), len(cols))
    sites = {(rows[k % len(rows)], cols[k % len(cols)]) for k in range(n)}
    sites |= {(0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)}
    return sorted(sites)


@pytest.mark.parametrize("shape", sorted(BLUR_SHAPES))
def test_blur_of_an_impulse_is_the_outer_product_of_the_weights(dev, ops, shape):
    H, W = shape
    s = _sigma(H, W)
    sites = _impulse_sites(H, W)
    x = torch.zeros((len(sites), H, W), dtype=torch.float32, device=dev)
    for k, (y, c) in enumerate(sites):
        x[k, y, c] = 1.0
    raw, mm = ops.gaussian_blur(x, s, normalize=False)
    _minmax_is_amin_amax(raw, mm)
    GH, GW = _G(H, s), _G(W, s)
    worst = 0.0
    for k, (y, c) in enumerate(sites):
        got = raw[k].cpu().numpy().astype(np.float64)
        want = np.outer(GH[:, y], GW[:, c])
        nz = want != 0
        assert not got[~nz].any(), "non-zero output outside the footprint of the impulse at %s" % ((y, c),)
        rel = np.abs(got[nz] - want[nz]) / want[nz]
        worst = max(worst, rel.max())
        assert rel.max() <= IMPULSE_REL, ((y, c), rel.max(), np.unravel_index(np.argmax(np.where(nz, np.abs(got - want) / np.where(nz, want, 1), 0)), got.shape))
    _observe("impulse %dx%d (%d sites, smallest product %.2g)" % (H, W, len(sites), gauss_weights(s).min() ** 2), worst, IMPULSE_REL)


@pytest.mark.parametrize("shape", BLUR_PLAIN_VS_TMA)
def test_plain_and_tma_vertical_passes_are_bit_identical(dev, ops, shape):
    H, W = shape
    s = _sigma(H, W)
    x = torch.from_numpy(_blur_maps(H, W)).to(dev)
    a, mma = ops.gaussian_blur(x, s, normalize=False)                 # 16-byte aligned: TMA vertical pass
    b, mmb = ops.gaussian_blur(_offset_view(x), s, normalize=False)   # 4-byte aligned: plain vertical pass
    assert torch.equal(a, b) and torch.equal(mma, mmb)
    an, _ = ops.gaussian_blur(x, s)
    bn, _ = ops.gaussian_blur(_offset_view(x), s)
    assert torch.equal(an, bn)


# ================================================================================================ B. threshold + upsample
UPSAMPLE_CASES = [  # P, H, W, rescale, with_background
    (21, 480, 640, False, True), (24, 427, 640, True, True), (21, 512, 683, True, True), (28, 375, 333, False, True),
    (32, 683, 512, True, False), (21, 427, 641, False, False), (21, 1848, 1848, True, True)]


def _class_maps(seed, B, C, P):
    cm = torch.stack([synth.saliency_maps(seed + b, C, P) for b in range(B)])
    cm[:, :, :3, :3] = 0            # a corner no class claims: the background is not empty
    return cm


@pytest.mark.parametrize("P,H,W,rescale,bg", UPSAMPLE_CASES)
def test_threshold_upsample_at_real_shapes(dev, ops, O, lib, P, H, W, rescale, bg):
    C = 5
    cm = _class_maps(P + H, 2, C, P)
    cm[1, 2] = 0                      # an all-zero class map: 0/0 -> NaN -> nothing kept (and a NaN channel when rescaled)
    out = ops.threshold_upsample(cm.to(dev), H, W, 0.15, rescale, bg)
    for b in range(2):
        with np.errstate(all="ignore"):
            ref = O.threshold_upsample(cm[b].clone(), 0.15, (H, W), rescale, bg).float()
        got = out[b].cpu()
        assert torch.equal(got.isnan(), ref.isnan())
        ok = ~ref.isnan()
        err = (got[ok].double() - ref[ok].double()).abs() - (1e-7 + 1e-5 * ref[ok].double().abs())
        assert err.max() <= 0
        if bg:
            assert torch.equal(got[0], ref[0])          # the background indicator is bit-exact
    # the scalar kernel through an output that is only 4-byte aligned: the same values bit for bit, nothing written outside
    Cc = C + (1 if bg else 0)
    n = 2 * Cc * H * W
    buf = torch.full((n + 2,), 12345.0, device=dev)
    ws_bytes = lib.pnp_threshold_upsample_workspace_bytes(2, C, P)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    cmd = cm.to(dev)
    rc = lib.pnp_threshold_upsample(cmd.data_ptr(), buf.data_ptr() + 4, ws.data_ptr(), ws_bytes, 2, C, P, H, W, 0.15, int(rescale),
                                    int(bg), torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    _same(buf[1:n + 1].view(out.shape), out)
    assert buf[0].item() == 12345.0 and buf[n + 1].item() == 12345.0


def test_threshold_upsample_one_class_quirk_at_a_large_shape(dev, ops, O):
    """With one class the reference's rescale silently does not happen (DRV:1079-1080)."""
    H, W = 1024, 1365
    cm = synth.saliency_maps(3, 1, 21)[None]
    out = ops.threshold_upsample(cm.to(dev), H, W, 0.15, True, True).cpu()
    ref = O.threshold_upsample(cm[0].clone(), 0.15, (H, W), True, True).float()
    assert torch.equal(out[0, 0], ref[0])
    assert ((out[0] - ref).abs() - (1e-7 + 1e-5 * ref.abs())).max() <= 0


# ================================================================================================ C. fused low-rank group
def _thresholded(cm, thr):
    """DRV:425-433 in float32 like the oracle: keep x where (x - min) / (max - min) >= thr."""
    out = cm.clone()
    for c in range(cm.shape[0]):
        with np.errstate(all="ignore"):
            th = (cm[c] - cm[c].min()) / (cm[c].max() - cm[c].min())
        out[c] = cm[c] * (th >= thr)
    return out


def _indicator(O, cm, thr, H, W, rescale):
    """The background indicator (DRV:446-450) as float64 [H, W]: the oracle's where it applies.  At H or W = 1 the oracle's
    squeeze() leaves a 2-D map, which it then treats as one class; there the same steps run on the unsqueezed [C, H, W]."""
    if min(H, W) > 1:
        with np.errstate(all="ignore"):
            return O.threshold_upsample(cm.clone(), thr, (H, W), rescale, True)[0].double().numpy()
    up = torch.nn.functional.interpolate(_thresholded(cm, thr)[None], size=(H, W), mode="bilinear", align_corners=True)[0]
    if rescale and cm.shape[0] > 1:
        f = up.view(cm.shape[0], -1)
        f -= f.min(-1, keepdim=True)[0]
        f /= f.max(-1, keepdim=True)[0]
    return (up.max(0)[0] == 0).double().numpy()


def _lowrank_ref(O, cm, H, W, rescale, bg, thr=0.15):
    """fp64 maps [C', H, W] after min/max normalisation: class c = A_H m_c A_W^T (A = G U), background = gaussian_filter of the
    oracle's indicator.  Returns (maps, unary [N, C'], labels [N])."""
    from scipy.ndimage import gaussian_filter
    C, P = cm.shape[0], cm.shape[-1]
    s = _sigma(H, W)
    m = _thresholded(cm, thr).double().numpy()
    AH, AW = _A(H, P, s), _A(W, P, s)
    chans = []
    if bg:
        chans.append(gaussian_filter(_indicator(O, cm, thr, H, W, rescale), s))
    chans += [AH @ m[c] @ AW.T for c in range(C)]
    maps = np.stack(chans)
    with np.errstate(all="ignore"):
        lo = maps.reshape(len(chans), -1).min(1)[:, None, None]
        hi = maps.reshape(len(chans), -1).max(1)[:, None, None]
        maps = (maps - lo) / (hi - lo)
        flat = maps.reshape(len(chans), -1)
        mx = flat.max(0)
        e = np.exp(flat - mx)
        sm = e / e.sum(0)
        unary = -np.log(np.clip(sm, 1e-5, 1.0)).T
    return maps, unary, np.argmax(maps.reshape(len(chans), -1), 0)


def _check_lowrank(out, b, maps, unary, labels, tag):
    Cc = maps.shape[0]
    got = out["maps"][b].cpu().numpy().astype(np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(maps))
    ok = ~np.isnan(maps)
    assert ok.any()
    err = np.abs(got[ok] - maps[ok]).max()
    _observe("lowrank maps " + tag, err, MAP_BOUND)
    assert err <= MAP_BOUND
    if "unary" in out:
        gu = out["unary"][b].cpu().numpy().astype(np.float64)
        assert np.array_equal(np.isnan(gu[:, :Cc]), np.isnan(unary))
        okU = ~np.isnan(unary)
        assert okU.any()
        errU = np.abs(gu[:, :Cc][okU] - unary[okU]).max()
        _observe("lowrank unary " + tag, errU, UNARY_BOUND)
        assert errU <= UNARY_BOUND
        assert not gu[:, Cc:].any()
    if "labels" in out and not np.isnan(maps).any():
        lab = out["labels"][b].cpu().numpy()
        srt = np.sort(maps.reshape(Cc, -1), 0)
        clear = (srt[-1] - srt[-2] > 2 * MAP_BOUND) if Cc > 1 else np.ones(lab.shape, bool)
        assert clear.any()
        assert np.array_equal(lab[clear], labels[clear])


def _lowrank_cases():
    combos = [(False, True), (True, True), (False, False), (True, False)]
    Ps = [p for p in LOWRANK_P if p > 1]
    cases = [(H, W, Ps[k % len(Ps)]) + combos[k % len(combos)] for k, (H, W) in enumerate(sorted(LOWRANK_SHAPES))]
    # the fused group's own background blur (indicator -> direct blur inside pnp_lowrank_blur_unary) at the largest shapes too
    return cases + [(H, W, P, rescale, True) for H, W, P, rescale, bg in cases[-2:] if not bg]


@pytest.mark.parametrize("H,W,P,rescale,bg", _lowrank_cases())
def test_lowrank_matches_the_fp64_closed_form(dev, ops, O, H, W, P, rescale, bg):
    B, C = 2, 5
    cm = _class_maps(1000 + P + W, B, C, P)
    out = ops.lowrank_blur_unary(cm.to(dev), H, W, 0.15, rescale, bg, _sigma(H, W), unary=True, labels=True, maps=True)
    for b in range(B):
        maps, unary, labels = _lowrank_ref(O, cm[b], H, W, rescale, bg)
        _check_lowrank(out, b, maps, unary, labels, "%dx%d P=%d" % (H, W, P))


@pytest.mark.parametrize("P", LOWRANK_P)
def test_lowrank_every_grid_size(dev, ops, O, P):
    H, W, C = 96, 80, 4
    cm = _class_maps(P, 1, C, P)
    if P == 1:
        cm = torch.rand(1, C, 1, 1, generator=torch.Generator().manual_seed(1))   # a 1x1 grid upsamples to a constant
    out = ops.lowrank_blur_unary(cm.to(dev), H, W, 0.15, True, True, _sigma(H, W), unary=True, labels=True, maps=True)
    maps, unary, labels = _lowrank_ref(O, cm[0], H, W, True, True)
    if P == 1:      # every map is constant: 0/0 = NaN everywhere, as in the reference
        assert bool(out["maps"].isnan().all()) and bool(out["unary"][0, :, :C + 1].isnan().all())
        return
    _check_lowrank(out, 0, maps, unary, labels, "P=%d" % P)


@pytest.mark.parametrize("H,W", LOWRANK_TINY)
@pytest.mark.parametrize("rescale", [False, True])
def test_lowrank_tiny_images(dev, ops, O, H, W, rescale):
    cm = _class_maps(H * 10 + W, 1, 3, 21)
    out = ops.lowrank_blur_unary(cm.to(dev), H, W, 0.15, rescale, True, _sigma(H, W), unary=True, labels=True, maps=True)
    maps, unary, labels = _lowrank_ref(O, cm[0], H, W, rescale, True)
    got = out["maps"][0].cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(maps))
    ok = ~np.isnan(maps)
    if ok.any():
        assert np.abs(got[ok] - maps[ok]).max() <= MAP_BOUND
    gu = out["unary"][0].cpu().numpy()
    assert np.array_equal(np.isnan(gu[:, :4]), np.isnan(unary))
    okU = ~np.isnan(unary)
    if okU.any():
        assert np.abs(gu[:, :4][okU] - unary[okU]).max() <= UNARY_BOUND
    # labels: numpy's argmax of the fp64 maps (the first NaN channel wins a NaN pixel) wherever the winner is clear
    flat = maps.reshape(4, -1)
    srt = np.sort(np.nan_to_num(flat, nan=np.inf), 0)
    with np.errstate(invalid="ignore"):
        clear = np.isnan(flat).any(0) | (srt[-1] - srt[-2] > 2 * MAP_BOUND)
    assert np.array_equal(out["labels"][0].cpu().numpy()[clear], labels[clear])


@pytest.mark.parametrize("C,H,W", [LOWRANK_WIDE_C, LOWRANK_HUGE_C])
def test_lowrank_many_classes(dev, ops, O, C, H, W):
    P = 21 if C < 300 else 32
    cm = _class_maps(C, 1, C, P)
    out = ops.lowrank_blur_unary(cm.to(dev), H, W, 0.15, False, True, _sigma(H, W), unary=True, labels=True, maps=True)
    maps, unary, labels = _lowrank_ref(O, cm[0], H, W, False, True)
    _check_lowrank(out, 0, maps, unary, labels, "C=%d %dx%d" % (C, H, W))


@pytest.mark.parametrize("H,W", [(480, 640), (683, 512)])
@pytest.mark.parametrize("rescale", [False, True])
def test_lowrank_padded_batch_equals_per_image_runs(dev, ops, H, W, rescale):
    counts = [1, 3, 2]
    Cmax = max(counts)
    cm = torch.full((len(counts), Cmax, 21, 21), float("nan"))
    for b, n in enumerate(counts):
        cm[b, :n] = _class_maps(50 + b, 1, n, 21)[0]
    nc = torch.tensor(counts, dtype=torch.int32, device=dev)
    out = ops.lowrank_blur_unary(cm.to(dev), H, W, 0.15, rescale, True, _sigma(H, W), unary=True, maps=True, n_classes=nc)
    lab = ops.lowrank_blur_unary(cm.to(dev), H, W, 0.15, rescale, True, _sigma(H, W), unary=False, labels=True, n_classes=nc)
    for b, n in enumerate(counts):
        ref = ops.lowrank_blur_unary(cm[b:b + 1, :n].contiguous().to(dev), H, W, 0.15, rescale, True, _sigma(H, W), unary=True,
                                     labels=True, maps=True)
        Cc = n + 1
        _same(out["unary"][b, :, :Cc], ref["unary"][0, :, :Cc])
        assert bool((out["unary"][b, :, Cc:] == float("inf")).all())
        _same(out["maps"][b, :Cc], ref["maps"][0])
        assert torch.equal(lab["labels"][b], ref["labels"][0])
        assert not bool(ref["unary"][0, :, :Cc].isnan().all())


# ================================================================================================ D. argmax and confusion
@pytest.mark.parametrize("C", ARGMAX_C)
@pytest.mark.parametrize("H,W", [CONFUSION_SHAPES[0][1:], CONFUSION_SHAPES[1][1:]])
def test_argmax_both_paths(dev, ops, C, H, W):
    B, N = 2, H * W
    rng = np.random.default_rng(C + N)
    x = rng.random((B, C, N)).astype(np.float32)
    x[0, 3, :500] = x[0, C - 1, :500] = 2.0       # ties: the first wins
    x[1, 5, 100:200] = np.nan                     # NaN counts as the maximum
    x[1, 2, 150:200] = np.nan                     # ... and the first NaN wins
    want = np.argmax(x, axis=1).astype(np.int32)
    xd = torch.from_numpy(x).to(dev)
    assert np.array_equal(ops.argmax_channels(xd).cpu().numpy(), want)
    assert np.array_equal(ops.argmax_channels(_offset_view(xd)).cpu().numpy(), want)


def _confusion_inputs(B, H, W, n_class, L=12):
    rng = np.random.default_rng(n_class * 31 + H)
    N = H * W
    gt = np.stack([synth.gt_labels(b + n_class, H, W, n_class) for b in range(B)]).reshape(B, N)
    k = rng.integers(0, N, (B, 64))
    for b in range(B):
        gt[b, k[b, :16]] = float(n_class)         # out of range
        gt[b, k[b, 16:32]] = -1.0                 # negative
        gt[b, k[b, 32:40]] = n_class - 0.5        # in range, truncates to n_class - 1
        gt[b, k[b, 40:48]] = 2.7                  # truncates to 2
        gt[b, k[b, 48:56]] = -0.25                # negative: outside the mask
    labels = rng.integers(0, L, (B, N)).astype(np.int32)
    lut = np.stack([rng.permutation(n_class)[:L] for _ in range(B)]).astype(np.int32)
    lut[::3, L - 1] = n_class                     # a label the dataset does not have: bad_count
    lut[1::3, L - 2] = -1
    return labels, gt.astype(np.float32), lut


def _confusion_ref(labels, gt, lut, n_class):
    pred = np.take_along_axis(lut, labels.astype(np.int64), 1)
    mask = (gt >= 0) & (gt < n_class)
    valid = mask & (pred >= 0) & (pred < n_class)
    hist = np.bincount((n_class * gt[valid].astype(np.int64) + pred[valid]).astype(np.int64), minlength=n_class * n_class)
    return hist.reshape(n_class, n_class).astype(np.int64), pred.astype(np.float32), int((mask & ~valid).sum())


def _run_confusion(ops, dev, labels, gt, lut, n_class, misaligned):
    lab_d, gt_d = torch.from_numpy(labels).to(dev), torch.from_numpy(gt).to(dev)
    pred = torch.full(gt.shape, -7.0, device=dev)
    if misaligned:
        lab_d, gt_d, pred = _offset_view(lab_d), _offset_view(gt_d), _offset_view(pred)
    hist = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    bad = torch.zeros((1,), dtype=torch.int32, device=dev)
    ops.confusion_accumulate(lab_d, gt_d, n_class, hist, lut=torch.from_numpy(lut).to(dev), pred_out=pred, bad_count=bad)
    return hist.cpu().numpy(), pred.cpu().numpy(), int(bad.item())


@pytest.mark.parametrize("n_class", CONFUSION_N_CLASS)
@pytest.mark.parametrize("B,H,W,misaligned", [s + (False,) for s in CONFUSION_SHAPES] + [CONFUSION_SHAPES[0] + (True,)])
def test_confusion_equals_bincount(dev, ops, n_class, B, H, W, misaligned):
    labels, gt, lut = _confusion_inputs(B, H, W, n_class)
    hist, pred, bad = _run_confusion(ops, dev, labels, gt, lut, n_class, misaligned)
    want, want_pred, want_bad = _confusion_ref(labels, gt, lut, n_class)
    assert np.array_equal(hist, want)
    assert np.array_equal(pred, want_pred)
    assert bad == want_bad and bad > 0


@pytest.mark.parametrize("n_class", [21, 171, 300])
@pytest.mark.parametrize("B,H,W", [CONFUSION_SHAPES[0], CONFUSION_SHAPES[1]])
def test_confusion_one_bin_for_every_pixel(dev, ops, n_class, B, H, W):
    """Every lane of every warp holds the same bin: the warp aggregation at its maximum (32 peers per atomic)."""
    N = H * W
    labels = np.zeros((B, N), np.int32)
    gt = np.full((B, N), 1.0, np.float32)
    lut = np.full((B, 1), 4, np.int32)
    hist, pred, bad = _run_confusion(ops, dev, labels, gt, lut, n_class, False)
    want = np.zeros((n_class, n_class), np.int64)
    want[1, 4] = B * N
    assert np.array_equal(hist, want) and bad == 0 and (pred == 4.0).all()


# ================================================================================================ E. limits and refusals
def test_1848_px_is_refused_where_the_direct_blur_runs(dev, ops):
    from pnp_ovss_b200 import PnpError, pipeline
    S = 1848
    with pytest.raises(PnpError):
        ops.gaussian_blur(torch.zeros((1, S, S), device=dev), _sigma(S, S))
    with pytest.raises(PnpError):
        ops.gaussian_blur(torch.zeros((1, S, 10), device=dev), _sigma(S, 10))
    cm = _class_maps(1, 1, 3, 21).to(dev)
    with pytest.raises(PnpError):
        ops.lowrank_blur_unary(cm, S, S, 0.15, False, True, _sigma(S, S))
    gts = torch.zeros((1, S, S), device=dev)
    guides = torch.zeros((1, S, S, 3), dtype=torch.uint8, device=dev)
    luts = torch.arange(4, dtype=torch.int32, device=dev)[None]
    hist = torch.zeros((21, 21), dtype=torch.int64, device=dev)
    for mode in ("blur", "blur+crf"):
        with pytest.raises(PnpError):
            pipeline.postprocess_batch(cm, guides, gts, luts, hist, threshold=0.15, rescale=False, with_background=True, mode=mode,
                                       n_class=21)
    assert not hist.any()
    with pytest.raises(PnpError):
        ops.gaussian_blur(torch.zeros((1, 10, 10), device=dev), 1024.2)          # radius 4097


def test_refusals_leave_caller_buffers_untouched(dev, lib):
    S, C, P = 1848, 3, 21
    st = torch.cuda.current_stream().cuda_stream
    x = torch.zeros((1, S, S), device=dev)
    out = torch.full((1, S, S), 12345.0, device=dev)
    mm = torch.full((1, 2), 12345.0, device=dev)
    ws = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
    assert lib.pnp_gaussian_blur(x.data_ptr(), out.data_ptr(), mm.data_ptr(), ws.data_ptr(), ws.numel(), 1, S, S, _sigma(S, S), 0,
                                 st) == PNP_ERR_INVALID_ARGUMENT
    cm = _class_maps(2, 1, C, P).to(dev)
    unary = torch.full((1, S * S, 4), 12345.0, device=dev)
    labels = torch.full((1, S * S), 777, dtype=torch.int32, device=dev)
    maps = torch.full((1, C + 1, S, S), 12345.0, device=dev)
    mmo = torch.full((C + 1, 2), 12345.0, device=dev)
    assert lib.pnp_lowrank_blur_unary(cm.data_ptr(), unary.data_ptr(), labels.data_ptr(), maps.data_ptr(), mmo.data_ptr(), ws.data_ptr(),
                                      ws.numel(), 1, C, P, S, S, 0.15, 0, 1, _sigma(S, S), st) == PNP_ERR_INVALID_ARGUMENT
    torch.cuda.synchronize()
    for t in (out, mm, unary, maps, mmo):
        assert bool((t == 12345.0).all())
    assert bool((labels == 777).all())


@pytest.mark.parametrize("H,W", LOWRANK_NO_BG_LARGE)
def test_lowrank_without_background_past_the_direct_blur_limit(dev, ops, O, H, W):
    """No background map, so no direct blur: only the fused kernels' own limits apply."""
    cm = _class_maps(H, 1, 3, 21)
    out = ops.lowrank_blur_unary(cm.to(dev), H, W, 0.15, True, False, _sigma(H, W), unary=True, labels=True, maps=True)
    maps, unary, labels = _lowrank_ref(O, cm[0], H, W, True, False)
    _check_lowrank(out, 0, maps, unary, labels, "no background %dx%d" % (H, W))


# ================================================================================================ F. non-finite inputs of the raw blur
@pytest.mark.parametrize("shape", [(480, 640), (512, 683)])
@pytest.mark.parametrize("value", [float("nan"), float("inf"), float("-inf")])
def test_non_finite_pixels_spread_like_scipy(dev, ops, shape, value):
    from scipy.ndimage import gaussian_filter
    H, W = shape
    s = _sigma(H, W)
    p = blur_plan(1, H, W, s)
    sites = [(p["v_rows"], p["h_groups"] * 16), (p["v_rows"] - 1, p["h_groups"] * 16 - 1), (0, W // 2), (H // 2, W - 1),
             (H - 1, 0)]
    rng = np.random.default_rng(H)
    x = rng.random((len(sites), H, W)).astype(np.float32)
    for k, (y, c) in enumerate(sites):
        x[k, y, c] = value
    raw, mm = ops.gaussian_blur(torch.from_numpy(x).to(dev), s, normalize=False)
    _minmax_is_amin_amax(raw, mm)
    raw = raw.cpu().numpy()
    for k in range(len(sites)):
        with np.errstate(all="ignore"):
            want = gaussian_filter(x[k].astype(np.float64), s)
        for pred in (np.isnan, np.isposinf, np.isneginf):
            assert np.array_equal(pred(raw[k]), pred(want)), (sites[k], pred.__name__, int(pred(raw[k]).sum()), int(pred(want).sum()))
        fin = np.isfinite(want)
        assert np.abs(raw[k][fin] - want[fin]).max() <= BLUR_ULP_BOUND(s, 1.0)


@pytest.mark.parametrize("shape", [(480, 640), (512, 683), (64, 48)])
def test_an_all_inf_map_reports_inf_inf(dev, ops, shape):
    H, W = shape
    x = torch.full((2, H, W), float("inf"), device=dev)
    x[1] = 0.5
    raw, mm = ops.gaussian_blur(x, _sigma(H, W), normalize=False)
    assert bool((raw[0] == float("inf")).all())
    assert mm[0].tolist() == [float("inf"), float("inf")]
    _minmax_is_amin_amax(raw, mm)
