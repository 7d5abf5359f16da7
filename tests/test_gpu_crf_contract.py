"""The dense-CRF kernels (pnp_ovss_b200/csrc/crf.cu, lattice.cu) against plain fp64 references and the sequential C
restatement (oracle/densecrf.c): every mean-field update variant the host planner can pick, the filter on both sides of the
blur-kernel switch, the lattice at the benchmark's batch size, the unary and the layout helpers.

Which update and blur kernel each channel count reaches is stated and checked in test_crf_algorithm.py, together with the fp64
operators and the bounds used here (each function's docstring gives its derivation).

Bounds.
- Q0 = softmax(-U), per element, within softmax_bound: Q_i (6 + 2 C) u + u of fp64 (u = 2^-24), from the exp error, the
  C - 1 additions of the sum and the division or reciprocal-multiply.
- Q1 (one iteration) against meanfield_step64 fed the GPU's own Q0 and lattice arrays (the lattice arrays are bit-exact
  against the restatement), so the bound covers one step's arithmetic only: softmax_bound with the exponent off by at most
  T = meanfield_exponent_bound, which adds up each message's relative error (L_k + 3 d_k + 7) u (L_k the longest vertex
  row) and the roundings of adding the messages to -U.  The bound is relative to Q_i, so a message error of a fraction of
  a percent (a dropped alpha is 20 %) fails it at every channel count.
- Labels are the first maximum of the GPU's own Q (NaN counts as the maximum) on every path, and the fp64 argmax wherever
  the fp64 leader's lead exceeds the two leaders' bounds.
- The filter (pnp_crf_filter) is bit-identical to the restatement, normalised or not; the lattice arrays too.
- The unary within unary_abs_bound of unary64: 16 u max|v| + (C + 27) u."""
import numpy as np
import pytest
import torch

from pnp_ovss_b200 import synthetic as synth
from test_crf_algorithm import (CRF_CP_CASES, crf_plan, features, is_fast_pair, meanfield_exponent_bound, messages64, softmax64,
                                softmax_bound, unary64, unary_abs_bound)

pytestmark = pytest.mark.gpu

B0, H0, W0 = 3, 37, 53          # partial 16x16 tiles, odd width
N0 = H0 * W0
WEIGHTS = {"spatial": 7.0, "bilateral": 10.0}
ORDERS = (("spatial", "bilateral"), ("bilateral", "spatial"))
FILTER_C = (5, 109, 112, 113, 150)
UNARY_C = (1, 2, 31, 32, 33, 64, 150, 171)
PACK_C = (1, 3, 4, 31, 32, 33, 65, 171)
OBSERVED = {}


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
def D():
    from oracle import densecrf
    densecrf.lib()
    return densecrf


def _np_lattice(lat):
    """The GPU lattice's arrays on the host, as the fp64 operators take them."""
    a = lat.arrays()
    return dict(offset=a["offset"].cpu().numpy(), bary=a["bary"].cpu().numpy(), nbr=a["nbr"].cpu().numpy(),
                norm=a["norm"].cpu().numpy(), M=lat.M, shared=bool(lat.struct.shared))


@pytest.fixture(scope="module")
def mf(dev, ops):
    """The mean-field cases' lattices: spatial (shared) and bilateral over B0 images of H0 x W0."""
    guides = np.stack([synth.guide_image(80 + b, H0, W0) for b in range(B0)])
    lats = {"spatial": ops.build_lattice(H0, W0, 3.0, device=dev),
            "bilateral": ops.build_lattice(H0, W0, 50.0, rgb=torch.from_numpy(guides).to(dev), srgb=5.0)}
    return lats, {k: _np_lattice(v) for k, v in lats.items()}


def _first_max(q):
    """numpy's argmax: the first maximum, a NaN counts as the maximum."""
    return np.argmax(q, -1)


def _check_q(key, q, ref, bound):
    err = np.abs(q - ref)
    worst = np.unravel_index(np.argmax(err / bound), err.shape)
    print("%s: max error %.3g, largest error / bound %.3g (error %.3g, bound %.3g at Q %.3g)"
          % (key, err.max(), err[worst] / bound[worst], err[worst], bound[worst], ref[worst]))
    assert (err <= bound).all(), key


def _check_labels(key, Q, labels, ref, bound):
    assert np.array_equal(labels, _first_max(Q)), key
    order = np.argsort(ref, -1)
    srt = np.take_along_axis(ref, order, -1)
    bsrt = np.take_along_axis(bound, order, -1)
    clear = srt[..., -1] - srt[..., -2] > bsrt[..., -1] + bsrt[..., -2] if ref.shape[-1] > 1 else np.ones(ref.shape[:-1], bool)
    assert clear.any(), key
    assert np.array_equal(labels[clear], np.argmax(ref, -1)[clear]), "%s: %d of %d clear labels differ" % (
        key, int((labels[clear] != np.argmax(ref, -1)[clear]).sum()), int(clear.sum()))


# ================================================================================================ mean-field update
@pytest.mark.parametrize("dc", [0, 3])
@pytest.mark.parametrize("Cp", CRF_CP_CASES)
def test_meanfield_update_every_branch(dev, ops, mf, Cp, dc):
    """Q0 and one iteration against fp64 for C = Cp (full last chunk) and Cp - 3 (one real channel in it), with both kernel
    orders: [spatial, bilateral] takes the folded fast path, [bilateral, spatial] the generic warp or block path.  Image 0
    has its last channel dead (unary +inf, as padded buckets mark a missing class), image 2 its first."""
    lats, lnp = mf
    C = Cp - dc
    if C < 1:
        pytest.skip("no channel left")
    rng = np.random.default_rng(Cp * 10 + dc)
    U = (rng.random((B0, N0, Cp)) ** 2 * 11.5).astype(np.float32)
    lead = rng.random((B0, N0)) < 0.5                 # half the pixels have a clear leader, whatever C is
    U[lead] += 2.0
    U[lead, rng.integers(0, C, int(lead.sum()))] = 0.25
    U[:, :, C:] = 0
    if C >= 2:
        U[0, :, C - 1] = np.inf
        U[2, :, 0] = np.inf
    Ug = torch.from_numpy(U).to(dev)
    Ur = U[..., :C]
    q0_ref = softmax64(-Ur)
    b0 = softmax_bound(q0_ref, C)
    q1_ref = bound1 = None
    for order in ORDERS:
        plan = crf_plan(Cp, B0, H0, W0)
        key = "Cp %d C %d [%s] %s%s" % (Cp, C, ",".join(order), plan["update"], " fast" if plan["warp"] and is_fast_pair(order) else "")
        L = [lats[k] for k in order]
        w = [WEIGHTS[k] for k in order]
        runs = {}
        for n_iter in (0, 1):
            Q, lab = ops.crf_inference(L, w, Ug, C, n_iter)
            if dc:     # padding channels are exactly 0, and NaN in their unary changes no bit
                assert float(Q[..., C:].abs().max()) == 0, key
                Un = Ug.clone()
                Un[..., C:] = float("nan")
                Qn, labn = ops.crf_inference(L, w, Un, C, n_iter)
                assert torch.equal(Qn, Q) and torch.equal(labn, lab), key
            runs[n_iter] = (Q[..., :C].double().cpu().numpy(), lab.cpu().numpy())
        q0, lab0 = runs[0]
        _check_q("Q0 " + key, q0, q0_ref, b0)
        _check_labels("labels0 " + key, q0, lab0, q0_ref, b0)
        if q1_ref is None:     # Q0 is the same for both orders (no kernel is applied), so is the fp64 step from it
            assert order == ORDERS[0]
            q0_first = q0
            lat_np = [lnp[k] for k in order]
            ys = messages64(q0, lat_np)
            t = -Ur.astype(np.float64)
            for wk, y in zip(w, ys):
                t = t + wk * y
            q1_ref = softmax64(t)
            bound1 = softmax_bound(q1_ref, C, meanfield_exponent_bound(Ur, ys, w, lat_np))
        else:
            assert np.array_equal(q0, q0_first), key
        q1, lab1 = runs[1]
        _check_q("Q1 " + key, q1, q1_ref, bound1)
        _check_labels("labels1 " + key, q1, lab1, q1_ref, bound1)
        if C >= 2:             # dead channels: exactly 0, never the label
            for q, lab in (runs[0], runs[1]):
                assert (q[0, :, C - 1] == 0).all() and (q[2, :, 0] == 0).all()
                assert not (lab[0] == C - 1).any() and not (lab[2] == 0).any()


@pytest.mark.parametrize("Cp", CRF_CP_CASES)
def test_meanfield_nan_row(dev, ops, mf, Cp):
    """At n_iter = 0 a NaN anywhere in a pixel's unary row makes its Q row NaN (padding stays 0) and its label 0, and leaves
    every other row as it was, bit for bit."""
    lats, _ = mf
    C = max(1, Cp - 3)
    rng = np.random.default_rng(Cp)
    U = torch.from_numpy((rng.random((B0, N0, Cp)) * 11.5).astype(np.float32)).to(dev)
    U[..., C:] = 0
    rows = [(0, 0, 0), (1, 777, C - 1), (2, N0 - 1, C // 2)]
    Un = U.clone()
    for b, p, c in rows:
        Un[b, p, c] = float("nan")
    for order in ORDERS:
        L = [lats[k] for k in order]
        w = [WEIGHTS[k] for k in order]
        Q, lab = ops.crf_inference(L, w, U, C, 0)
        Qn, labn = ops.crf_inference(L, w, Un, C, 0)
        hit = torch.zeros((B0, N0), dtype=torch.bool, device=dev)
        for b, p, _ in rows:
            hit[b, p] = True
            assert bool(Qn[b, p, :C].isnan().all()) and bool((Qn[b, p, C:] == 0).all())
            assert int(labn[b, p]) == 0
        assert torch.equal(Qn[~hit], Q[~hit]) and torch.equal(labn[~hit], lab[~hit])


# ================================================================================================ filter
def _filter_case(D, H, W, C, seed):
    img = synth.guide_image(seed, H, W)
    crf = D.DenseCRF2D(W, H, C)
    crf.addPairwiseGaussian(3, 7)
    crf.addPairwiseBilateral(50, 5, img, 10)
    x = np.random.default_rng(seed).random((C, H * W)).astype(np.float32)
    return img, crf, x


@pytest.mark.parametrize("C", FILTER_C)
def test_filter_bit_exact_both_blur_kernels(dev, ops, D, C):
    """Cp 8, 112, 112, 116, 152: both sides of the two-axis blur switch at Cp = 112."""
    img, crf, x = _filter_case(D, H0, W0, C, C)
    assert crf_plan(ops.crf_pad_channels(C))["blur"] == ("axis2" if C <= 112 else "axis")
    xg = ops.crf_pack(torch.from_numpy(x[None]).to(dev))
    for k, lat in enumerate((ops.build_lattice(H0, W0, 3.0, device=dev),
                             ops.build_lattice(H0, W0, 50.0, rgb=torch.from_numpy(img[None]).to(dev), srgb=5.0))):
        y = ops.crf_unpack(ops.crf_filter(lat, xg), C)[0].cpu().numpy()
        assert np.array_equal(y, crf.kernel_apply(k, x)), (C, k)


@pytest.mark.parametrize("C", [5, 150])
def test_filter_unnormalised_is_lattice_compute(dev, ops, D, C):
    img = synth.guide_image(C + 1, H0, W0)
    x = np.random.default_rng(C).random((H0 * W0, C)).astype(np.float32)
    xg = ops.crf_pack(torch.from_numpy(np.ascontiguousarray(x.T[None])).to(dev))
    for f, lat in ((features(H0, W0, 3.0), ops.build_lattice(H0, W0, 3.0, device=dev)),
                   (features(H0, W0, 50.0, img, 5.0), ops.build_lattice(H0, W0, 50.0, rgb=torch.from_numpy(img[None]).to(dev), srgb=5.0))):
        y = ops.crf_filter(lat, xg, normalized=False)[0, :, :C].cpu().numpy()
        assert np.array_equal(y, D.Lattice(f).compute(x)), C


@pytest.mark.parametrize("C", [5, 150])
def test_filter_shared_lattice_over_ten_images(dev, ops, D, C):
    """B = 10 > 8: the shared lattice's grid is split over min(B, 8) image rows."""
    Bn = 10
    crf = D.DenseCRF2D(W0, H0, C)
    crf.addPairwiseGaussian(3, 7)
    x = np.random.default_rng(C).random((Bn, C, N0)).astype(np.float32)
    lat = ops.build_lattice(H0, W0, 3.0, device=dev)
    y = ops.crf_unpack(ops.crf_filter(lat, ops.crf_pack(torch.from_numpy(x).to(dev))), C).cpu().numpy()
    for b in range(Bn):
        assert np.array_equal(y[b], crf.kernel_apply(0, x[b])), b


def test_filter_batched_bilateral_at_cp_152(dev, ops, D):
    C, Bn = 150, 3
    imgs = np.stack([synth.guide_image(90 + b, H0, W0) for b in range(Bn)])
    x = np.random.default_rng(9).random((Bn, C, N0)).astype(np.float32)
    lat = ops.build_lattice(H0, W0, 50.0, rgb=torch.from_numpy(imgs).to(dev), srgb=5.0)
    y = ops.crf_unpack(ops.crf_filter(lat, ops.crf_pack(torch.from_numpy(x).to(dev))), C).cpu().numpy()
    for b in range(Bn):
        crf = D.DenseCRF2D(W0, H0, C)
        crf.addPairwiseBilateral(50, 5, imgs[b], 10)
        assert np.array_equal(y[b], crf.kernel_apply(0, x[b])), b


def test_filter_one_bench_image(dev, ops, D):
    H = W = 336
    C = 21
    img, crf, x = _filter_case(D, H, W, C, 336)
    xg = ops.crf_pack(torch.from_numpy(x[None]).to(dev))
    for k, lat in enumerate((ops.build_lattice(H, W, 3.0, device=dev),
                             ops.build_lattice(H, W, 50.0, rgb=torch.from_numpy(img[None]).to(dev), srgb=5.0))):
        y = ops.crf_unpack(ops.crf_filter(lat, xg), C)[0].cpu().numpy()
        assert np.array_equal(y, crf.kernel_apply(k, x)), k


# ================================================================================================ lattice at bench size
def _check_slice(a, ref, norm, base, lp0, n):
    assert np.array_equal(a["offset"][lp0:lp0 + n], ref.offset + base)
    assert np.array_equal(a["bary"][lp0:lp0 + n], ref.barycentric)
    nb = a["nbr"][:, base:base + ref.M]
    assert np.array_equal(nb[:, :, 0], np.where(ref.n1 < 0, 0, ref.n1 + 1 + base))
    assert np.array_equal(nb[:, :, 1], np.where(ref.n2 < 0, 0, ref.n2 + 1 + base))
    assert np.array_equal(a["norm"][lp0:lp0 + n], norm)


def _check_csr(a, M):
    """row_ptr / csr_pix / csr_w / csr_norm are the entries grouped by vertex, in entry (= pixel) order."""
    off = a["offset"].ravel()
    D1 = a["offset"].shape[1]
    rp = a["row_ptr"]
    assert rp[0] == 0 and rp[-1] == off.size and rp.size == M + 1
    assert np.array_equal(np.diff(rp), np.bincount(off, minlength=M))
    order = np.argsort(off, kind="stable")
    assert np.array_equal(a["csr_pix"], order // D1)
    assert np.array_equal(a["csr_w"], a["bary"].ravel()[order])
    assert np.array_equal(a["csr_norm"], a["norm"][order // D1])


def test_bilateral_lattice_at_bench_size(dev, ops, D):
    """configs[1]: 35 images of 336^2, d = 5: 23.7 M entries, 5 789 scan blocks, so the scan spine carries 6 times.  Every
    image's slice of the lattice against the restatement, and the CSR over the whole batch."""
    Bn, H, W = 35, 336, 336
    N = H * W
    imgs = np.stack([synth.guide_image(200 + b, H, W) for b in range(Bn)])
    lat = ops.build_lattice(H, W, 50.0, rgb=torch.from_numpy(imgs).to(dev), srgb=5.0)
    assert -(-N * Bn * 6 // 4096) == 5789
    a = {k: v.cpu().numpy() for k, v in lat.arrays().items()}
    base = 0
    for b in range(Bn):
        ref = D.Lattice(features(H, W, 50.0, imgs[b], 5.0))
        crf = D.DenseCRF2D(W, H, 1)
        crf.addPairwiseBilateral(50, 5, imgs[b], 10)
        _check_slice(a, ref, crf.kernel_norm(0), base, b * N, N)
        base += ref.M
    assert lat.M == base
    _check_csr(a, lat.M)


@pytest.mark.parametrize("side", [336, 512])
def test_spatial_lattice_at_full_size(dev, ops, D, side):
    lat = ops.build_lattice(side, side, 3.0, device=dev)
    a = {k: v.cpu().numpy() for k, v in lat.arrays().items()}
    ref = D.Lattice(features(side, side, 3.0))
    crf = D.DenseCRF2D(side, side, 1)
    crf.addPairwiseGaussian(3, 7)
    assert lat.M == ref.M
    _check_slice(a, ref, crf.kernel_norm(0), 0, 0, side * side)
    _check_csr(a, lat.M)


# ================================================================================================ unary and layout
@pytest.mark.parametrize("C", UNARY_C)
def test_unary_from_maps(dev, ops, C):
    """C <= 32: one pass through a shared-memory tile; C > 32: statistics pass, then 32-channel slabs.  N = 1 961 is not a
    multiple of the 128-pixel tile."""
    Bn = 3
    rng = np.random.default_rng(C)
    for with_minmax in (False, True):
        maps = (rng.random((Bn, C, N0)) * (1.0 if with_minmax else 30.0)).astype(np.float32)
        maps[1, C // 2, 100] = np.nan                     # a NaN column: the pixel's whole row is NaN
        mm = None
        if with_minmax:
            mm = np.stack([np.nanmin(maps, -1), np.nanmax(maps, -1)], -1).reshape(Bn * C, 2).astype(np.float32)
        Ug = ops.crf_unary_from_maps(torch.from_numpy(maps).to(dev), None if mm is None else torch.from_numpy(mm).to(dev))
        got = Ug.cpu().numpy()
        Cp = ops.crf_pad_channels(C)
        assert got.shape == (Bn, N0, Cp) and (got[..., C:] == 0).all()
        want = unary64(maps, mm)
        assert np.array_equal(np.isnan(got[..., :C]), np.isnan(want))
        assert np.isnan(got[1, 100, :C]).all()
        ok = ~np.isnan(want)
        vmax = 1.0 if with_minmax else 30.0
        bound = unary_abs_bound(vmax, C)
        err = np.abs(got[..., :C][ok] - want[ok]).max()
        _observe("unary C %d minmax %d" % (C, with_minmax), err, bound)
        assert err <= bound


@pytest.mark.parametrize("C", PACK_C)
def test_pack_unpack_round_trip(dev, ops, C):
    Bn = 3
    x = torch.randn(Bn, C, N0, device=dev)
    x[0, 0, 0] = float("nan")
    x[1, C - 1, N0 - 1] = float("-inf")
    p = ops.crf_pack(x)
    Cp = ops.crf_pad_channels(C)
    want = torch.zeros(Bn, N0, Cp, device=dev)
    want[..., :C] = x.transpose(1, 2)
    assert torch.equal(p.nan_to_num(7.0), want.nan_to_num(7.0)) and bool(p[0, 0, 0].isnan())
    back = ops.crf_unpack(p, C)
    assert torch.equal(back.nan_to_num(7.0), x.nan_to_num(7.0)) and bool(back[0, 0, 0].isnan())
