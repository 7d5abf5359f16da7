"""GPU parity tests: every CUDA entry point (through the C ABI) against the CPU oracle on the same seeded inputs,
against the committed golden fixtures, and -- at BASELINE.json sizes -- through size-independent properties.

Tolerances (north_star): integer / index / label work bit-exact; floating point within 1e-3 relative.  Where the
kernels follow the oracle's fp32 operation order the tests ask for bit equality."""
import numpy as np
import pytest
import torch

import synth
from make_golden_cases import DRIVER_CASES, MERGE_CASES, VOC_NMS

pytestmark = pytest.mark.gpu

RTOL = 1e-3  # north_star: "within 1e-3 relative (fp32 accumulate)"


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def O():
    from oracle import hotpath
    return hotpath


@pytest.fixture(scope="module")
def ops():
    from pnp_ovss_b200 import ops as _ops
    return _ops


def _close(a, b, rtol=RTOL, atol=1e-7):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape
    assert np.array_equal(np.isnan(a), np.isnan(b))
    m = ~np.isnan(a)
    err = np.abs(a[m] - b[m]) - (atol + rtol * np.abs(b[m]))
    assert (err <= 0).all(), "max violation %g (max abs diff %g)" % (err.max(), np.abs(a[m] - b[m]).max())


# ------------------------------------------------------------------------------------------------ (a)
@pytest.mark.parametrize("K", [442, 785, 1025, 33])
def test_softmax_fwd(dev, ops, O, K):
    g = torch.Generator().manual_seed(K)
    s = torch.randn(3, 12, 7, K, generator=g) * 8
    ref = O.cross_attention_probs(s, None, head_size=64)
    out = ops.softmax_fwd(s.to(dev), None, 0.125)
    _close(out.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=1e-12)
    mask = torch.zeros(3, K)
    mask[:, -5:] = -10000.0
    ref = O.cross_attention_probs(s, mask.view(3, 1, 1, K), head_size=64)
    out = ops.softmax_fwd(s.to(dev), mask.to(dev), 0.125)
    _close(out.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=1e-12)
    assert torch.allclose(out.sum(-1).cpu(), torch.ones(3, 12, 7), atol=1e-5)


def test_softmax_fwd_golden(dev, ops, golden):
    s = torch.from_numpy(golden["gc_scores_scaled"]).to(dev)
    out = ops.softmax_fwd(s.contiguous(), None, 1.0)
    _close(out.cpu().numpy(), golden["gc_probs"], rtol=1e-5, atol=1e-12)


@pytest.mark.parametrize("K,T", [(442, 9), (785, 5)])
def test_softmax_bwd_gradcam(dev, ops, O, K, T):
    g = torch.Generator().manual_seed(7 * K + T)
    B, h = 4, 12
    probs = torch.softmax(torch.randn(B, h, T, K, generator=g), -1)
    dprobs = torch.randn(B, h, T, K, generator=g) * 1e-3
    mask = torch.zeros(B, 500, dtype=torch.int64)
    for b in range(B):
        mask[b, :T - b] = 1
    P = int(round((K - 1) ** 0.5))
    ref_cam = O.gradcam_head(probs, dprobs, mask, P, 9)
    ref_ds = O.softmax_backward(probs, dprobs)
    ds, cam = ops.softmax_bwd_gradcam(probs.to(dev), dprobs.to(dev), mask.to(dev), 9, 0.125, True, True)
    assert np.array_equal(cam.cpu().numpy().reshape(ref_cam.shape), ref_cam.numpy())  # same products, same order
    _close(ds.cpu().numpy(), ref_ds.numpy(), rtol=1e-4, atol=1e-10)
    ds2, cam2 = ops.softmax_bwd_gradcam(probs.to(dev), dprobs.to(dev), mask.to(dev), 9, 0.125, False, True)
    assert ds2 is None and torch.equal(cam2, cam)
    ds3, cam3 = ops.softmax_bwd_gradcam(probs.to(dev), dprobs.to(dev), None, 0, 0.125, True, False)
    assert cam3 is None and torch.equal(ds3, ds)


def test_gradcam_golden(dev, ops, golden):
    probs = torch.from_numpy(golden["gc_probs"]).to(dev)
    dprobs = torch.from_numpy(golden["gc_dprobs"]).to(dev)
    m500 = torch.from_numpy(golden["gc_mask500"]).to(dev)
    for head in (9, 0):
        _, cam = ops.softmax_bwd_gradcam(probs, dprobs, m500, head, 0.5, False, True)
        want = golden["gc_head%d" % head]
        assert np.array_equal(cam.cpu().numpy().reshape(want.shape), want)


def test_softmax_autograd_function_matches_torch(dev):
    """The autograd.Function used inside the model's block-8 cross-attention: forward and both gradients."""
    from pnp_ovss_b200.blip_itm import FusedXattnSoftmax, GradcamCapture
    g = torch.Generator().manual_seed(5)
    B, h, T, K = 2, 12, 6, 442
    s = torch.randn(B, h, T, K, generator=g).to(dev).requires_grad_(True)
    v = torch.randn(B, h, K, 64, generator=g).to(dev)
    mask = torch.ones(B, 500, dtype=torch.int64, device=dev)
    cap = GradcamCapture(head=9, token_mask=mask)
    p = FusedXattnSoftmax.apply(s, None, 0.125, cap)
    loss = (p @ v).square().sum()
    loss.backward()
    s2 = s.detach().clone().requires_grad_(True)
    p2 = torch.softmax(s2 * 0.125, -1)
    p2.retain_grad()
    ((p2 @ v).square().sum()).backward()
    _close(p.detach().cpu().numpy(), p2.detach().cpu().numpy(), rtol=1e-5, atol=1e-12)
    _close(s.grad.cpu().numpy(), s2.grad.cpu().numpy(), rtol=1e-3, atol=1e-6)
    want = (p2.detach()[:, 9, 1:, 1:] * p2.grad[:, 9, 1:, 1:].clamp(0))
    _close(cap.gradcam.cpu().numpy(), want.cpu().numpy(), rtol=1e-4, atol=1e-9)


# ------------------------------------------------------------------------------------------------ (b)
def test_token_merge_golden(dev, ops, O, golden):
    from pnp_ovss_b200 import host
    tok = synth.SyntheticWordPieceTokenizer()
    for class_lists in MERGE_CASES.values():
        for cl in class_lists:
            tok("A picture of " + " ".join(cl))
    for name, class_lists in MERGE_CASES.items():
        ids = golden["merge_%s_ids" % name]
        g = torch.from_numpy(golden["merge_%s_g" % name]).to(dev)
        B = len(class_lists)
        Cmax = max(len(c) for c in class_lists)
        start = np.zeros((B, Cmax), np.int32)
        length = np.zeros((B, Cmax), np.int32)
        div = np.ones((B, Cmax), np.float32)
        for b, cl in enumerate(class_lists):
            segs = host.build_token_segments(host.token_strings(ids[b], tok.decode), len(cl))
            for c, (s, l, d) in enumerate(segs):
                start[b, c], length[b, c], div[b, c] = s, l, d
        out = ops.token_merge(g, torch.from_numpy(start).to(dev), torch.from_numpy(length).to(dev), torch.from_numpy(div).to(dev))
        for b, cl in enumerate(class_lists):
            assert np.array_equal(out[b, :len(cl)].cpu().numpy(), golden["merge_%s_out%d" % (name, b)]), (name, b)


# ------------------------------------------------------------------------------------------------ (c)
def _gpu_dropout(dev, fn, rows, imgs, R, P):
    from pnp_ovss_b200.pipeline import salience_dropout_loop
    x = imgs.clone().to(dev)
    return salience_dropout_loop(lambda t: fn(t.cpu(), rows).to(dev), x, None, R, P), x


def test_dropout_loop_golden(dev, golden):
    imgs = torch.from_numpy(golden["drop_imgs"])
    rows = torch.from_numpy(golden["drop_rows"])
    T = int(golden["drop_T"])
    B, P = imgs.shape[0], 6
    for R in (1, 4):
        fn = synth.SynthGradcamFn(21, B, T, P)
        (g0, agg, chosen), _ = _gpu_dropout(dev, fn, rows, imgs, R, P)
        assert np.array_equal(g0.cpu().numpy(), golden["drop_R%d_g0" % R])
        if R > 1:
            assert np.array_equal(agg.cpu().numpy(), golden["drop_R%d_agg" % R])
            assert chosen.shape == (B, 10 * R) and int(chosen.min()) >= 0


@pytest.mark.parametrize("P,S", [(21, 336), (28, 448)])
def test_dropout_loop_vs_oracle(dev, O, P, S):
    B, T, R = 3, 9, 4
    g = torch.Generator().manual_seed(P)
    imgs = torch.randn(B, 3, S, S, generator=g)
    rows = torch.ones(B, T - 1)
    rows[1, -2:] = 0  # a shorter caption: its SEP row stays in the score (quirk a4)
    fn_o = synth.SynthGradcamFn(3, B, T, P)
    g0_o, agg_o, chosen_o, dropped_o = O.salience_dropout(lambda x: fn_o(x, rows), imgs, R, P, argsort_kind="stable")
    fn_g = synth.SynthGradcamFn(3, B, T, P)
    (g0, agg, chosen), x = _gpu_dropout(dev, fn_g, rows, imgs, R, P)
    assert np.array_equal(g0.cpu().numpy(), g0_o.numpy())
    assert np.array_equal(agg.cpu().numpy(), agg_o.numpy())
    ch = chosen.cpu().numpy()
    for b in range(B):
        for r in range(R):  # same set per round (order inside a round is ascending score in both)
            assert sorted(ch[b, 10 * r:10 * r + 10].tolist()) == sorted(chosen_o[b][10 * r:10 * r + 10]), (b, r)
    # after the last round the image carries every chosen block zeroed (the reference re-zeroes at the next round start)
    want = dropped_o[-1].clone()
    for b in range(B):
        for idx in chosen_o[b][-10:]:
            want[b, :, (idx // P) * 16:(idx // P) * 16 + 16, (idx % P) * 16:(idx % P) * 16 + 16] = 0
    assert torch.equal(x.cpu(), want)


# ------------------------------------------------------------------------------------------------ (d)
@pytest.mark.parametrize("rescale", [False, True])
@pytest.mark.parametrize("bg", [False, True])
@pytest.mark.parametrize("shape", [(21, 336, 336), (21, 375, 500), (28, 97, 131)])
def test_threshold_upsample(dev, ops, O, rescale, bg, shape):
    P, H, W = shape
    C = 5
    maps = torch.stack([synth.saliency_maps(10 + i, C, P) for i in range(2)])
    maps[1, 2] = 0  # an all-zero class map: 0/0 min-max -> NaN -> nothing kept (and NaN channel when rescaled)
    out = ops.threshold_upsample(maps.to(dev), H, W, 0.15, rescale, bg).cpu()
    for b in range(2):
        with np.errstate(all="ignore"):
            ref = O.threshold_upsample(maps[b].clone(), 0.15, (H, W), rescale, bg).float()
        _close(out[b].numpy(), ref.numpy(), rtol=1e-5, atol=1e-7)
        if bg:
            assert np.array_equal(out[b, 0].numpy(), ref[0].numpy())  # the background mask is bit-exact


def test_threshold_upsample_single_class(dev, ops, O):
    maps = synth.saliency_maps(3, 1, 21).unsqueeze(0)
    out = ops.threshold_upsample(maps.to(dev), 120, 160, 0.15, True, True).cpu()
    ref = O.threshold_upsample(maps[0].clone(), 0.15, (120, 160), True, True).float()
    _close(out[0].numpy(), ref.numpy(), rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("shape", [(336, 336), (375, 500), (64, 48), (20, 30), (512, 512), (10, 200), (200, 12), (1, 64)])
def test_gaussian_blur_vs_scipy(dev, ops, O, shape):
    H, W = shape
    rng = np.random.default_rng(H * 1000 + W)
    x = rng.random((3, H, W)).astype(np.float32)
    x[1] = (x[1] > 0.7).astype(np.float32)  # a binary map like the background channel
    sigma = 0.05 * max(H, W)
    out, mm = ops.gaussian_blur(torch.from_numpy(x).to(dev), sigma, normalize=True)
    raw, mm2 = ops.gaussian_blur(torch.from_numpy(x).to(dev), sigma, normalize=False)
    from scipy.ndimage import gaussian_filter
    for i in range(3):
        # raw blur: fp32 accumulation over up to 205 taps against scipy's float64 accumulators
        _close(raw[i].cpu().numpy(), gaussian_filter(x[i], sigma), rtol=5e-6, atol=1e-7)
        # after (y-min)/(max-min) the same absolute error is divided by the map's dynamic range (tiny for iid noise),
        # so the normalised map is compared at 1e-3 relative plus 1e-4 of its unit range
        ref = O.blurring(torch.from_numpy(x[i]), (H, W))
        _close(out[i].cpu().numpy(), ref, rtol=RTOL, atol=1e-4)
    assert torch.equal(mm, mm2)
    assert torch.allclose(raw.amin((1, 2)), mm[:, 0]) and torch.allclose(raw.amax((1, 2)), mm[:, 1])


def test_gaussian_blur_golden(dev, ops, golden):
    for tag in ("a", "b"):
        x = golden["blur_%s_in" % tag]
        out, _ = ops.gaussian_blur(torch.from_numpy(x).to(dev).unsqueeze(0), 0.05 * max(x.shape), normalize=True)
        _close(out[0].cpu().numpy(), golden["blur_%s_out" % tag], rtol=RTOL, atol=2e-6)


def test_gaussian_blur_constant_map_is_nan(dev, ops):
    """A constant map blurs to a constant: (y-min)/(max-min) = 0/0 = NaN everywhere, like the reference (DRV:1151-1152)."""
    x = torch.zeros(1, 64, 64, device=dev)
    out, _ = ops.gaussian_blur(x, 3.2, normalize=True)
    assert bool(torch.isnan(out).all())


# ------------------------------------------------------------------------------------------------ (f)
@pytest.mark.parametrize("n_class", [21, 183, 300])
def test_confusion_matrix(dev, ops, O, n_class):
    rng = np.random.default_rng(n_class)
    B, H, W = 3, 120, 97
    gt = np.stack([synth.gt_labels(5 + b, H, W, n_class) for b in range(B)])
    gt[0, :3, :3] = -1.0
    gt[1, 0, 0] = float(n_class)
    labels = rng.integers(0, 7, (B, H * W)).astype(np.int32)
    lut = np.stack([rng.permutation(n_class)[:7] for _ in range(B)]).astype(np.int32)
    hist = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    pred = torch.empty((B, H * W), dtype=torch.float32, device=dev)
    ops.confusion_accumulate(torch.from_numpy(labels).to(dev), torch.from_numpy(gt).view(B, -1).to(dev), n_class, hist,
                             lut=torch.from_numpy(lut).to(dev), pred_out=pred)
    want = np.zeros((n_class, n_class), dtype=np.int64)
    for b in range(B):
        p = lut[b][labels[b]]
        want += O.fast_hist(gt[b].flatten(), p.astype(np.float32), n_class)
        assert np.array_equal(pred[b].cpu().numpy(), p.astype(np.float32))
    assert np.array_equal(hist.cpu().numpy(), want)


def test_confusion_golden(dev, golden):
    from pnp_ovss_b200 import reference_api as R
    n = int(golden["hist_n"])
    gt, pred = golden["hist_gt"], golden["hist_pred"]
    assert np.array_equal(R._fast_hist(gt.flatten(), pred.flatten(), n), golden["hist_out"])
    table, hist = R.scores([gt, gt.T.copy()], [pred, pred.T.copy()], None, n)
    assert np.array_equal(hist, golden["scores_hist"])
    assert table["Mean IoU"] == float(golden["scores_miou"])
    # with the category table the drivers pass, 'Class IoU' is the reference's dict keyed by name (DRV:1130-1137)
    cats = {i: "class_%d" % i for i in range(1, n)}
    named, _ = R.scores([gt, gt.T.copy()], [pred, pred.T.copy()], cats, n)
    assert list(named["Class IoU"]) == ["Background"] + ["class_%d" % i for i in range(1, n)]
    assert np.array_equal(np.array(list(named["Class IoU"].values())), table["Class IoU"], equal_nan=True)


def test_salience_dropout_round_rejects_misshapen_buffers(dev, ops):
    """The kernel writes agg / ensemble_r / norm_imgs unconditionally: wrong layouts must be refused, not written out of bounds."""
    from pnp_ovss_b200 import PnpError
    B, Tm, P, patch = 2, 6, 4, 16
    g = torch.rand(B, Tm, P, P, device=dev)
    chosen = torch.full((B, 20), -1, dtype=torch.int32, device=dev)
    imgs = torch.zeros(B, 3, P * patch, P * patch, device=dev)
    ok = dict(agg=torch.empty_like(g), chosen=chosen, n_prev=0, imgs=imgs, norm_imgs=torch.zeros(B, P * patch, P * patch, 3, device=dev),
              P=P, patch=patch, row_lo=3, row_hi=Tm - 1, save_len=10, round_idx=0)
    ops.salience_dropout_round(g, **ok)
    for bad in (dict(norm_imgs=torch.zeros(B, 3, P * patch, P * patch, device=dev)), dict(agg=torch.empty(B, Tm - 1, P, P, device=dev)),
                dict(ensemble_r=torch.empty(B, Tm, P, P - 1, device=dev)), dict(chosen=torch.full((B - 1, 20), -1, dtype=torch.int32, device=dev)),
                dict(chosen=torch.full((B, 5), -1, dtype=torch.int32, device=dev))):
        with pytest.raises(PnpError):
            ops.salience_dropout_round(g, **dict(ok, **bad))


def test_argmax_channels(dev, ops):
    rng = np.random.default_rng(0)
    for N in (336 * 336, 1001):
        x = rng.random((2, 21, N)).astype(np.float32)
        x[0, 3, :50] = x[0, 7, :50] = 2.0     # ties: first wins
        x[1, 5, 10:20] = np.nan               # NaN counts as the maximum
        x[1, 2, 15:20] = np.nan               # ... and the first NaN wins
        out = ops.argmax_channels(torch.from_numpy(x).to(dev)).cpu().numpy()
        assert np.array_equal(out, np.argmax(x, axis=1).astype(np.int32))


# ------------------------------------------------------------------------------------------------ error behaviour
def test_ops_fail_loudly_on_bad_arguments(dev, ops):
    """No silent fallbacks: wrong dtypes / layouts / shapes / undersized workspaces raise PnpError (negative ABI code)."""
    import ctypes
    from pnp_ovss_b200 import PnpError, _lib
    with pytest.raises(PnpError):
        ops.softmax_fwd(torch.zeros(1, 12, 4, 442, dtype=torch.float16, device=dev))
    with pytest.raises(PnpError):
        ops.softmax_fwd(torch.zeros(1, 12, 4, 2000, device=dev))                    # K beyond the register-row limit
    with pytest.raises(PnpError):
        ops.argmax_channels(torch.zeros(2, 3, 16, device=dev).transpose(1, 2))      # not contiguous
    with pytest.raises(PnpError):
        ops.gaussian_blur(torch.zeros(1, 8, 8, device=dev), 0.0)                    # sigma must be positive
    with pytest.raises(PnpError):
        ops.threshold_upsample(torch.zeros(1, 2, 40, 40, device=dev), 64, 64, 0.15, False, True)   # P*P > 1024
    lat = ops.build_lattice(16, 16, 3.0, rgb=torch.zeros(2, 16, 16, 3, dtype=torch.uint8, device=dev), srgb=5.0)
    with pytest.raises(PnpError):
        ops.crf_filter(lat, torch.zeros(3, 256, 4, device=dev))                     # lattice built for 2 images, 3 given
    lib = _lib.load()
    x = torch.zeros(1, 8, 8, device=dev)
    y = torch.empty_like(x)
    mm = torch.empty(1, 2, device=dev)
    ws = torch.empty(16, dtype=torch.uint8, device=dev)
    rc = lib.pnp_gaussian_blur(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), ctypes.c_void_p(mm.data_ptr()),
                               ctypes.c_void_p(ws.data_ptr()), 16, 1, 8, 8, 1.0, 1, ctypes.c_void_p(0))
    assert rc == -2 and b"workspace" in lib.pnp_error_string(rc)                    # PNP_ERR_WORKSPACE
    hist = torch.zeros(3, 3, dtype=torch.int64, device=dev)
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    ops.confusion_accumulate(torch.full((1, 4), 7, dtype=torch.int32, device=dev), torch.zeros(1, 4, device=dev), 3, hist, bad_count=bad)
    assert int(bad.item()) == 4 and int(hist.sum()) == 0                            # out-of-range ids are counted, never binned


# ------------------------------------------------------------------------------------------------ (f)1 GEMM operand kernels
def _split_ref(t):
    hi = ((t.view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)
    return torch.cat([hi, t - hi, hi], -1)


@pytest.mark.parametrize("M,K", [(1, 4), (37, 768), (442 * 3, 1024), (50, 4096)])
def test_tf32_split3_is_exact(dev, ops, M, K):
    """[hi | lo | hi]: hi has no bits below TF32's mantissa, hi + lo == x bit for bit (integer work: exact)."""
    x = (torch.randn(M, K, generator=torch.Generator().manual_seed(M + K)) * 3).to(dev)
    got = ops.tf32_split3(x)
    assert got.shape == (M, 3 * K)
    assert torch.equal(got, _split_ref(x))
    assert int((got[:, :K].view(torch.int32) & 0x1FFF).abs().max()) == 0
    assert torch.equal(got[:, :K] + got[:, K:2 * K], x)
    special = torch.tensor([[0.0, -0.0, float("inf"), -float("inf")], [3.4028234e38, -3.4028234e38, 1e-45, float("nan")]], device=dev)
    s3 = ops.tf32_split3(special)
    back = s3[:, :4] + s3[:, 4:8]
    assert torch.equal(back[~special.isnan()], special[~special.isnan()]) and bool(back[1, 3].isnan())


@pytest.mark.parametrize("K", [768, 1024, 2048])
def test_layernorm_tf32_split3_matches_torch(dev, ops, K):
    g = torch.Generator().manual_seed(K)
    M = 333
    x, res = torch.randn(M, K, generator=g).to(dev) * 2 + 0.3, torch.randn(M, K, generator=g).to(dev)
    gamma, beta, rb = (torch.randn(K, generator=g).to(dev) for _ in range(3))
    want = torch.nn.functional.layer_norm(x.double(), (K,), gamma.double(), beta.double(), 1e-6)
    s3, plain = ops.layernorm_tf32_split3(x.clone(), gamma, beta, 1e-6, split=True, plain=True)
    _close(plain.cpu(), want.cpu(), rtol=1e-5, atol=2e-6)
    assert torch.equal(s3, _split_ref(plain))
    # fused residual: x <- x + res + bias (written back in place), then the same LayerNorm
    xin = x.clone()
    s3, plain = ops.layernorm_tf32_split3(xin, gamma, beta, 1e-6, residual=res, residual_bias=rb, split=True, plain=True)
    assert torch.equal(xin, (x + res) + rb)
    want = torch.nn.functional.layer_norm(xin.double(), (K,), gamma.double(), beta.double(), 1e-6)
    _close(plain.cpu(), want.cpu(), rtol=1e-5, atol=2e-6)
    assert torch.equal(s3, _split_ref(plain))


def test_gelu_tf32_split3_matches_torch(dev, ops):
    g = torch.Generator().manual_seed(9)
    x, b = torch.randn(257, 4096, generator=g).to(dev) * 3, torch.randn(4096, generator=g).to(dev)
    got = ops.gelu_tf32_split3(x, b)
    want = torch.nn.functional.gelu((x + b).double())
    back = got[:, :4096] + got[:, 4096:8192]
    _close(back.cpu(), want.cpu(), rtol=1e-5, atol=1e-6)
    assert torch.equal(got[:, :4096], got[:, 8192:])
    assert int((got[:, :4096].view(torch.int32) & 0x1FFF).abs().max()) == 0


def test_tripled_tf32_gemm_is_fp32_grade(dev, ops):
    """One TF32 GEMM over [x_hi|x_lo|x_hi] x [W_hi|W_hi|W_lo]^T against an fp64 product: the error must be of the order of
    a native fp32 GEMM's, far below plain TF32's."""
    from pnp_ovss_b200.blip_itm import _mm3, _w3
    g = torch.Generator().manual_seed(2)
    x, w, b = torch.randn(512, 1024, generator=g).to(dev), (torch.randn(768, 1024, generator=g) * 0.02).to(dev), torch.randn(768, generator=g).to(dev)
    truth = torch.nn.functional.linear(x.double(), w.double(), b.double())
    err3 = (_mm3(ops.tf32_split3(x), _w3(w), b).double() - truth).abs().max().item()
    err32 = (torch.nn.functional.linear(x, w, b).double() - truth).abs().max().item()
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    err_tf32 = (torch.nn.functional.linear(x, w, b).double() - truth).abs().max().item()
    torch.backends.cuda.matmul.allow_tf32 = prev
    assert err3 <= 4 * err32 + 1e-6, (err3, err32)
    assert err3 * 20 <= err_tf32, (err3, err_tf32)


# ------------------------------------------------------------------------------------------------ (d) fused low-rank group
def _oracle_blurred_maps(O, cm, thr, H, W, rescale, with_bg):
    """DRV:424-455 then DRV:1005-1011 on the CPU: threshold, torch bilinear upsample, [Scale_0_1], background, scipy blur + min-max."""
    with np.errstate(all="ignore"):
        x = O.threshold_upsample(cm.clone(), thr, (H, W), rescale, with_bg)
        return O.blur_channels(x.float(), (H, W)).numpy()


LOWRANK_CASES = [  # C, P, H, W, rescale, with_background
    (3, 21, 336, 336, False, True), (20, 21, 336, 336, True, True), (5, 21, 333, 500, False, False), (2, 24, 384, 384, True, True),
    (7, 28, 448, 448, False, True), (4, 32, 512, 512, True, False), (1, 21, 100, 75, True, True), (9, 21, 500, 375, True, True)]


@pytest.mark.parametrize("C,P,H,W,rescale,with_bg", LOWRANK_CASES)
def test_lowrank_blur_matches_the_reference_chain(dev, ops, O, C, P, H, W, rescale, with_bg):
    """One fused launch group against the reference's own chain (torch interpolate + scipy gaussian_filter + min-max): the
    normalised blurred maps within 5e-6, the per-channel (min, max) of the raw blur, the CRF unary and the blur-only labels."""
    B = 2
    cms = torch.stack([synth.saliency_maps(100 * C + b + P, C, P) for b in range(B)])
    out = ops.lowrank_blur_unary(cms.to(dev), H, W, 0.15, rescale, with_bg, 0.05 * max(H, W), unary=True, labels=True, maps=True, minmax=True)
    Cc = C + (1 if with_bg else 0)
    assert out["maps"].shape == (B, Cc, H, W) and out["unary"].shape == (B, H * W, (Cc + 3) // 4 * 4)
    for b in range(B):
        want = _oracle_blurred_maps(O, cms[b], 0.15, H, W, rescale, with_bg)
        got = out["maps"][b].cpu().numpy()
        assert np.array_equal(np.isnan(got), np.isnan(want))
        ok = ~np.isnan(want)
        assert np.abs(got[ok] - want[ok]).max() <= 5e-6, np.abs(got[ok] - want[ok]).max()
        # unary = -log(clip(softmax_c, 1e-5, 1)) of those maps (DRV:1057-1063), pixel-major, padding channels zero
        with np.errstate(all="ignore"):
            sm = torch.softmax(torch.from_numpy(want), 0).numpy()
            U = -np.log(np.clip(sm, 1e-5, 1.0)).reshape(Cc, H * W).T
        gotU = out["unary"][b].cpu().numpy()
        assert np.array_equal(np.isnan(gotU[:, :Cc]), np.isnan(U))
        okU = ~np.isnan(U)      # (with Scale_0_1 and many classes the background channel is empty -> 0/0 -> every unary is NaN)
        assert not okU.any() or np.abs(gotU[:, :Cc][okU] - U[okU]).max() <= 3e-5
        assert not gotU[:, Cc:].any()
        # blur-only labels: argmax of the normalised maps; a handful of pixels may sit on a numerical tie
        lab = out["labels"][b].cpu().numpy().reshape(H, W)
        if not np.isnan(want).any():
            assert (lab != want.argmax(0)).mean() <= 2e-4
            srt = np.sort(want, 0)
            clear = (srt[-1] - srt[-2] > 1e-4) if Cc > 1 else np.ones((H, W), bool)
            assert np.array_equal(lab[clear], want.argmax(0)[clear])          # wherever the winner is clear the label is exact
    # background indicator: bit-exact wherever the direct kernels' upsample says so (it is the same arithmetic)
    if with_bg:
        direct = ops.threshold_upsample(cms.to(dev), H, W, 0.15, rescale, True)
        blurred, mm = ops.gaussian_blur(direct[:, :1].contiguous(), 0.05 * max(H, W), normalize=False)
        got_mm = out["minmax"].view(B, Cc, 2)[:, 0]
        assert torch.equal(got_mm, mm.view(B, 2))


def test_lowrank_blur_equals_the_direct_kernels(dev, ops):
    """The fused path against the direct one (pnp_threshold_upsample -> pnp_gaussian_blur -> pnp_crf_unary_from_maps) at the
    benchmark shape: same unary within 3e-5 -- the two differ only in fp32 summation order."""
    B, C, P, S = 3, 20, 21, 336
    cms = torch.stack([synth.saliency_maps(7 + b, C, P) for b in range(B)])
    cms[:, :, :5, :5] = 0     # a corner no class claims: the background channel is not empty (an empty one is 0/0 = NaN everywhere)
    cms = cms.to(dev)
    for rescale in (False, True):
        out = ops.lowrank_blur_unary(cms, S, S, 0.15, rescale, True, 0.05 * S, unary=True, maps=True)
        x = ops.threshold_upsample(cms, S, S, 0.15, rescale, True)
        xb, mm = ops.gaussian_blur(x, 0.05 * S, normalize=False)
        U = ops.crf_unary_from_maps(xb.view(B, C + 1, S * S), mm)
        assert torch.equal(out["unary"].isnan(), U.isnan())
        assert torch.nan_to_num(out["unary"] - U).abs().max().item() <= 3e-5
        xn, _ = ops.gaussian_blur(x, 0.05 * S, normalize=True)
        assert torch.equal(out["maps"].isnan(), xn.isnan())
        assert torch.nan_to_num(out["maps"] - xn).abs().max().item() <= 5e-6
        if not rescale:
            assert not bool(U.isnan().any())        # the comparison is not vacuous


def test_lowrank_blur_nan_and_single_class_quirks(dev, ops, O):
    """A class whose map is constant thresholds to all zeros (0/0 -> NaN -> False, DRV:425-433): its blurred channel is 0/0 = NaN
    (DRV:1151-1152), the unary of every channel of those pixels is NaN and argmax picks the first NaN channel -- as in the
    reference chain.  With one class Scale_0_1 silently does not happen (DRV:1079-1080)."""
    P, S = 21, 96
    cm = synth.saliency_maps(5, 3, P)
    cm[1] = 0.25                                    # constant -> dropped class
    out = ops.lowrank_blur_unary(cm[None].to(dev), S, S, 0.15, True, True, 0.05 * S, unary=True, labels=True, maps=True)
    want = _oracle_blurred_maps(O, cm, 0.15, S, S, True, True)
    got = out["maps"][0].cpu().numpy()
    assert np.isnan(want[2]).all() and np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert ok.any() and np.abs(got[ok] - want[ok]).max() <= 5e-6
    assert bool(out["unary"][0, :, :4].isnan().all()) and not out["unary"][0, :, 4:].any()
    first_nan = int(np.isnan(want).all(axis=(1, 2)).argmax())
    assert bool((out["labels"][0] == first_nan).all())      # numpy/torch argmax: the (first) NaN channel wins
    one = synth.saliency_maps(6, 1, P)
    out1 = ops.lowrank_blur_unary(one[None].to(dev), S, S, 0.15, True, True, 0.05 * S, unary=False, maps=True)
    want1 = _oracle_blurred_maps(O, one, 0.15, S, S, True, True)
    assert np.abs(out1["maps"][0].cpu().numpy() - want1).max() <= 5e-6


def test_lowrank_blur_rejects_bad_arguments(dev, ops):
    from pnp_ovss_b200 import PnpError
    cm = torch.zeros(1, 2, 33, 33, device=dev)
    with pytest.raises(PnpError):
        ops.lowrank_blur_unary(cm, 64, 64, 0.15, False, True, 3.2)            # P > 32
    with pytest.raises(PnpError):
        ops.lowrank_blur_unary(torch.zeros(1, 2, 21, 21, device=dev), 64, 64, 0.15, False, True, 0.0)   # sigma must be positive
    with pytest.raises(PnpError):
        ops.lowrank_blur_unary(torch.zeros(1, 2, 21, 21), 64, 64, 0.15, False, True, 3.2)               # CPU tensor


# ------------------------------------------------------------------------------------------------ 3xFP16 operand kernels
def _split16_ref(t, hi_scale=1.0):
    h = t.half()
    l = ((t - h.float()) * 2048.0).half()
    return torch.cat([(h.float() * hi_scale).half(), l, h], -1)


@pytest.mark.parametrize("M,K,hi_scale", [(1, 4, 1.0), (37, 768, 1.0), (442 * 3, 1024, 8.0), (50, 4096, 1.0)])
def test_fp16_split3_is_exact(dev, ops, M, K, hi_scale):
    """[h*2^a | (x-h)*2^11 | h]: bit-equal to the torch restatement; h + l 2^-11 reproduces x to 2^-22 relative."""
    x = (torch.randn(M, K, generator=torch.Generator().manual_seed(M + K)) * 3).to(dev)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    got = ops.fp16_split3(x, 1.0, hi_scale, flag)
    assert got.dtype == torch.float16 and got.shape == (M, 3 * K)
    assert torch.equal(got, _split16_ref(x, hi_scale)) and int(flag.item()) == 0
    back = got[:, 2 * K:].double() + got[:, K:2 * K].double() / 2048.0
    assert ((back - x.double()).abs() <= 2.0 ** -21 * x.double().abs() + 1e-10).all()      # (+ fp16's subnormal floor for tiny |x|)
    scaled = ops.fp16_split3(x, 0.25, hi_scale, flag)                      # in_scale: the split of x/4, exactly
    assert torch.equal(scaled, _split16_ref(x * 0.25, hi_scale))
    big = x.clone()
    big[0, 0] = 70000.0                                                    # beyond fp16: the flag is raised, nothing else
    ops.fp16_split3(big, 1.0, hi_scale, flag)
    assert int(flag.item()) == 1


def test_fused_fp16_producers_match_torch(dev, ops):
    g = torch.Generator().manual_seed(11)
    M, K = 200, 1024
    x, res = torch.randn(M, K, generator=g).to(dev) * 2 + 0.3, torch.randn(M, K, generator=g).to(dev) * 2048.0
    gamma, beta, rb = (torch.randn(K, generator=g).to(dev) for _ in range(3))
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    xin = x.clone()
    s3, plain = ops.layernorm_fp16_split3(xin, gamma, beta, 1e-6, residual=res, residual_scale=1.0 / 2048.0, residual_bias=rb, hi_scale=1.0,
                                          split=True, plain=True, flag=flag)
    want_x = x + res / 2048.0 + rb
    _close(xin.cpu(), want_x.cpu(), rtol=1e-6, atol=1e-6)
    want = torch.nn.functional.layer_norm(xin.double(), (K,), gamma.double(), beta.double(), 1e-6)
    _close(plain.cpu(), want.cpu(), rtol=1e-5, atol=2e-6)
    assert torch.equal(s3, _split16_ref(plain)) and int(flag.item()) == 0
    f, b = torch.randn(64, 4096, generator=g).to(dev) * 3 * 2048.0, torch.randn(4096, generator=g).to(dev)
    got = ops.gelu_fp16_split3(f, b, 1.0 / 2048.0, 1.0, flag)
    want = torch.nn.functional.gelu((f / 2048.0 + b).double())
    back = got[:, 8192:].double() + got[:, 4096:8192].double() / 2048.0
    _close(back.cpu(), want.cpu(), rtol=1e-5, atol=1e-6)


def test_tripled_fp16_gemm_is_fp32_grade(dev, ops):
    """One fp16 GEMM over [x_h|x_l|x_h] x [W_h 2^11|W_h|W_l]^T (fp32 accumulate) against an fp64 product: an error of the order
    of a native fp32 GEMM's, far below a plain fp16 product's."""
    from pnp_ovss_b200.blip_itm import FP16_OUT_SCALE, _mm16, _w16
    g = torch.Generator().manual_seed(2)
    x, w = torch.randn(512, 1024, generator=g).to(dev), (torch.randn(768, 1024, generator=g) * 0.02).to(dev)
    truth = x.double() @ w.double().t()
    w16, hi_scale = _w16(w)
    assert hi_scale == 1.0                                       # realistic weights leave the activations their full fp16 range
    y = _mm16(ops.fp16_split3(x, 1.0, hi_scale), w16) / FP16_OUT_SCALE
    err3 = (y.double() - truth).abs().max().item()
    err32 = (x @ w.t()).double().sub(truth).abs().max().item()
    err16 = (x.half() @ w.half().t()).double().sub(truth).abs().max().item()
    assert err3 <= 12 * err32 + 1e-6, (err3, err32)              # tensor-core accumulation truncates: a few times native fp32
    assert err3 * 30 <= err16, (err3, err16)
    wbig = w.clone()
    wbig[0, 0] = 100.0                                           # a weight above 32 moves part of the 2^11 to the activation side
    w16b, hi_b = _w16(wbig)
    assert hi_b == 4.0 and bool(torch.isfinite(w16b.float()).all())
    yb = _mm16(ops.fp16_split3(x, 1.0, hi_b), w16b) / FP16_OUT_SCALE
    assert (yb.double() - x.double() @ wbig.double().t()).abs().max().item() <= 1e-4 * 100


# ------------------------------------------------------------------------------------------------ encoder attention (3xFP16)
@pytest.mark.parametrize("B,L,H", [(2, 442, 16), (1, 785, 4), (3, 64, 2), (1, 37, 1)])
def test_attention_fp16x3_is_fp32_grade(dev, ops, B, L, H):
    """softmax(Q K^T / 8) V on the fp16 tensor cores with hi/lo-split operands against an fp64 evaluation: error of the order
    of torch's own fp32 attention, two orders of magnitude below a plain fp16 attention; ragged L (tail tiles) included."""
    g = torch.Generator().manual_seed(L + H)
    qkv = (torch.randn(B, L, 3, H, 64, generator=g) * torch.tensor([2.0, 2.0, 1.0]).view(1, 1, 3, 1, 1)).to(dev)
    q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    truth = torch.nn.functional.scaled_dot_product_attention(q.double(), k.double(), v.double()).permute(0, 2, 1, 3).reshape(B, L, H * 64)
    got = ops.attention_fp16x3(qkv)
    ref32 = torch.nn.functional.scaled_dot_product_attention(q, k, v).permute(0, 2, 1, 3).reshape(B, L, H * 64)
    ref16 = torch.nn.functional.scaled_dot_product_attention(q.half(), k.half(), v.half()).float().permute(0, 2, 1, 3).reshape(B, L, H * 64)
    sc = truth.abs().max().item()
    e_got, e32, e16 = ((t.double() - truth).abs().max().item() / sc for t in (got, ref32, ref16))
    print("attention L=%d: max err / max |o|: 3xfp16 kernel %.2e, torch fp32 %.2e, plain fp16 %.2e" % (L, e_got, e32, e16))
    assert e_got <= 20 * e32 + 1e-6 and e_got * 30 <= e16
    # the form the encoder uses: operands carrying the 3xFP16 GEMM's factor 2^11
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    got_scaled = ops.attention_fp16x3((qkv * 2048.0).contiguous(), in_scale=1.0 / 2048.0, flag=flag)
    assert torch.equal(got_scaled, got) and int(flag.item()) == 0
    # ... and the fused operand split of the output is the split kernel's, bit for bit
    flag.zero_()
    got3 = ops.attention_fp16x3(qkv, flag=flag, split_hi_scale=2.0)
    assert torch.equal(got3, ops.fp16_split3(got, 1.0, 2.0, flag)) and int(flag.item()) == 0
    ops.attention_fp16x3((qkv * 1e6).contiguous(), flag=flag)            # out of fp16's range: the flag says so
    assert int(flag.item()) == 1


@pytest.mark.parametrize("B,L,H", [(1, 1, 1), (2, 64, 3), (1, 129, 2), (3, 442, 4), (1, 1000, 1)])
def test_attention_fp16x3_tile_edges(dev, ops, B, L, H):
    """At the edges of the 64-key and 128-row tiles (L = 1, 64, 129, 1000): deterministic, within 4e-6 of an fp64 evaluation (rows
    past L / keys past L never leak in), and the operand-split output is the split of the kernel's own fp32 output."""
    g = torch.Generator().manual_seed(17 * L + H)
    qkv = torch.randn(B, L, 3, H, 64, generator=g).to(dev)
    q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    truth = torch.nn.functional.scaled_dot_product_attention(q.double(), k.double(), v.double()).permute(0, 2, 1, 3).reshape(B, L, H * 64)
    got = ops.attention_fp16x3(qkv)
    got2 = ops.attention_fp16x3(qkv)
    sc = truth.abs().max().item()
    assert torch.equal(got, got2)
    assert (got.double() - truth).abs().max().item() / sc <= 4e-6
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    assert torch.equal(ops.attention_fp16x3(qkv, flag=flag, split_hi_scale=4.0), ops.fp16_split3(got, 1.0, 4.0, flag))
    assert int(flag.item()) == 0
