"""The host planner of pnp_crf_inference (pnp_ovss_b200/csrc/crf.cu) restated in Python, the fp64 operators the dense-CRF
contract tests build their references from, and the lattice shape limit.  test_gpu_crf_contract.py takes its channel counts,
its references and its bounds from here.

The planner picks the mean-field update kernel from Cp, the padded channel count: LPP lanes per pixel x CPL chunks per lane
(the split of the Cp/4 float4 chunks over a warp that idles the fewest lanes, ties to more chunks per lane), the register-capped
occ3 entry point when CPL is 4 or 6 and there are at least 12 chunks, and the block kernel past Cp = 768.  Separately, the
splat/blur runs two lattice axes per launch up to Cp = 112 and one above.  CRF_CP_CASES reaches every combination that any Cp
in 4..1024 reaches.

The fp64 operators take the lattice arrays themselves (offset, bary, nbr with 0 as the sentinel, norm), so a GPU test can feed
them the GPU's own lattice and bound the arithmetic of one operation.  Below they are checked against the sequential C
restatement in oracle/densecrf.c."""
import ctypes

import numpy as np
import pytest
import torch

from pnp_ovss_b200 import synthetic as synth

U32 = 2.0 ** -24
PNP_OK, PNP_ERR_INVALID_ARGUMENT = 0, -1

# ----------------------------------------------------------------------------------------------- planner of pnp_crf_inference
CRF_CP_CASES = [4, 8, 12, 16, 20, 24, 28, 36, 40, 44, 52, 84, 112, 116, 152, 172, 768, 772, 1024]


def crf_plan(Cp, B=1, H=37, W=53):
    """The update kernel and blur kernel pnp_crf_inference launches for B images of H x W at Cp channels."""
    nch = Cp // 4
    LPP = CPL = 0
    best = 0.0
    for cpl in (1, 2, 3, 4, 6):
        lpp = -(-nch // cpl)
        if lpp > 32:
            continue
        eff = float(32 // lpp) * nch / (32.0 * cpl)
        if eff >= best - 1e-9:                      # ties: more chunks per lane wins
            best, LPP, CPL = eff, lpp, cpl
    occ3 = CPL in (4, 6) and nch >= 12
    warp = CPL > 0 and W > 0 and B * H * W < (1 << 31) // Cp
    update = ("cpl%d%s" % (CPL, "_occ3" if occ3 else "")) if warp else "block"
    return dict(LPP=LPP, CPL=CPL, occ3=occ3, warp=warp, update=update, blur="axis2" if Cp <= 112 else "axis")


def crf_branch(Cp):
    """(update kernel, more than one lane per pixel, blur kernel): what a mean-field case exercises."""
    p = crf_plan(Cp)
    return p["update"], p["warp"] and p["LPP"] > 1, p["blur"]


def is_fast_pair(kernels):
    """kFast (folded weights, FMA, __expf) is used for [spatial shared, bilateral batched] only."""
    return len(kernels) == 2 and kernels[0] == "spatial" and kernels[1] == "bilateral"


def test_the_cp_cases_reach_every_branch():
    every = {crf_branch(Cp) for Cp in range(4, 1025, 4)}
    assert {crf_branch(Cp) for Cp in CRF_CP_CASES} == every
    assert {b[0] for b in every} == {"cpl1", "cpl2", "cpl3", "cpl4", "cpl4_occ3", "cpl6", "cpl6_occ3", "block"}
    assert ("cpl4_occ3", True, "axis2") in every and ("cpl4_occ3", True, "axis") in every


@pytest.mark.parametrize("Cp,LPP,CPL,occ3", [(4, 1, 1, False), (20, 5, 1, False), (12, 1, 3, False), (36, 3, 3, False),
                                             (16, 1, 4, False), (28, 2, 4, False), (52, 4, 4, True), (124, 8, 4, True),
                                             (24, 1, 6, False), (44, 2, 6, False), (84, 4, 6, True), (768, 32, 6, True)])
def test_planner_choices(Cp, LPP, CPL, occ3):
    p = crf_plan(Cp)
    assert (p["LPP"], p["CPL"], p["occ3"], p["warp"]) == (LPP, CPL, occ3, True)


def test_planner_edges():
    assert crf_plan(768)["update"] == "cpl6_occ3" and crf_plan(772)["update"] == "block"
    assert crf_plan(112)["blur"] == "axis2" and crf_plan(116)["blur"] == "axis"
    # bench batch (configs[1]: 35 images of 336^2, 21 classes -> Cp 24) and padded buckets of 8-15 classes + background
    assert crf_plan(24, 35, 336, 336)["update"] == "cpl6"
    assert crf_plan(12)["update"] == "cpl3" and crf_plan(16)["update"] == "cpl4"
    assert not crf_plan(1024, 1 << 20, 1, 1)["warp"]          # B N >= 2^31 / Cp: block kernel


# ----------------------------------------------------------------------------------------------- fp64 operators
def lattice_alpha(d):
    """1 / (1 + 2^-d) rounded to fp32, as the restatement and the kernels slice with."""
    return float(np.float32(1.0) / (np.float32(1.0) + np.float32(2.0 ** -d)))


def splat_blur_slice64(lat, x):
    """K x in float64 (un-normalised): x [n_lp, C] over the lattice's pixels -> [n_lp, C].  lat: offset [n_lp, d+1],
    bary [n_lp, d+1], nbr [d+1, M, 2] (vertex + 1, 0 = none), M.  As sparse matrices over the vertex rows (row 0 is the
    sentinel and stays 0): the splat S adds bary-weighted pixels into their d+1 vertices, each axis blur is
    v + 1/2 (v[n1] + v[n2]), and the slice is alpha S^T."""
    import scipy.sparse as sp
    offset, bary, nbr = np.asarray(lat["offset"]), np.asarray(lat["bary"], np.float64), np.asarray(lat["nbr"])
    n_lp, D1 = offset.shape
    M = int(lat["M"])
    S = sp.csr_matrix((bary.ravel(), ((offset + 1).ravel(), np.repeat(np.arange(n_lp), D1))), shape=(M + 1, n_lp))
    v = S @ np.asarray(x, np.float64)
    rows = np.arange(1, M + 1)
    for j in range(D1):
        n1, n2 = nbr[j, :M, 0], nbr[j, :M, 1]
        r = np.concatenate([rows, rows[n1 > 0], rows[n2 > 0]])
        c = np.concatenate([rows, n1[n1 > 0], n2[n2 > 0]])
        w = np.concatenate([np.ones(M), np.full(int((n1 > 0).sum()) + int((n2 > 0).sum()), 0.5)])
        v = sp.csr_matrix((w, (r, c)), shape=(M + 1, M + 1)) @ v
    return (S.T @ v) * lattice_alpha(D1 - 1)


def filter64(lat, x, normalized=True):
    """norm . K (norm . x) (or K x) for x [B, N, C]: a shared lattice filters every image, a batched one the whole batch."""
    B, N, C = x.shape
    x = np.asarray(x, np.float64)
    if lat["shared"]:
        return np.stack([filter64(dict(lat, shared=False), x[b:b + 1], normalized)[0] for b in range(B)])
    xs = x.reshape(B * N, C)
    if not normalized:
        return splat_blur_slice64(lat, xs).reshape(B, N, C)
    nrm = np.asarray(lat["norm"], np.float64)[:, None]
    return (nrm * splat_blur_slice64(lat, nrm * xs)).reshape(B, N, C)


def softmax64(t):
    """softmax over the last axis; a NaN anywhere in a row makes the row NaN, a -inf entry gets exactly 0."""
    t = np.asarray(t, np.float64)
    with np.errstate(invalid="ignore"):
        e = np.exp(t - t.max(-1, keepdims=True))
        return e / e.sum(-1, keepdims=True)


def messages64(Q, lattices):
    return [filter64(lat, Q, normalized=True) for lat in lattices]


def meanfield_step64(U, Q, lattices, weights):
    """softmax(-U + sum_k w_k norm_k . K_k (norm_k . Q)); U, Q [B, N, C]."""
    t = -np.asarray(U, np.float64)
    for w, y in zip(weights, messages64(Q, lattices)):
        t = t + w * y
    return softmax64(t)


def unary64(maps, minmax=None):
    """pnp_crf_unary_from_maps in float64: maps [B, C, N] (normalised by minmax [B*C, 2] when given) -> softmax over C ->
    clip to [1e-5, 1] -> -log, as [B, N, C].  A NaN in any channel of a pixel makes its whole row NaN."""
    B, C, N = maps.shape
    v = np.asarray(maps, np.float64)
    if minmax is not None:
        mm = np.asarray(minmax, np.float64).reshape(B, C, 2)
        with np.errstate(invalid="ignore", divide="ignore"):
            v = (v - mm[:, :, 0, None]) / (mm[:, :, 1, None] - mm[:, :, 0, None])
    p = softmax64(np.moveaxis(v, 1, 2))
    with np.errstate(invalid="ignore"):
        return -np.log(np.clip(p, 1e-5, 1.0))


# ----------------------------------------------------------------------------------------------- error bounds
def max_row(lat):
    """Longest vertex row: the most terms one splat sum adds."""
    return int(np.bincount(np.asarray(lat["offset"]).ravel(), minlength=int(lat["M"])).max())


def filter_rel_bound(L, d, normalized):
    """Relative error of the fp32 splat/blur/slice of a non-negative field, given exact lattice arrays and norm.  Every
    intermediate is a sum of non-negative products, so relative errors add along the longest chain of roundings: the splat
    (the norm product, the weight product, L - 1 additions), 2 per blur axis, the slice (weight and alpha products, d
    additions) and the final norm product.  First order, with 1 % for the higher-order terms."""
    n = (L + 1) + 2 * (d + 1) + (d + 2) + 1 if normalized else L + 2 * (d + 1) + (d + 2)
    return 1.01 * n * U32


def softmax_bound(q_ref, C, T=0.0):
    """|Q_gpu - Q64| per element, for an fp32 softmax of C channels whose exponents are within T of fp64's.  Exact
    arithmetic on exponents off by T moves Q_i by at most Q_i (e^{2T} - 1).  Then max subtraction and exp (expf's 2 ulp, or
    __expf's 2 + 1.16 |x| ulp) give e_i a relative error of at most (2 + 2.2 |x_i|) u; the sum adds C - 1 roundings and, as
    e^x |x| <= 1/e, at most (2 + 0.81 (C - 1)) u through its terms; the division or reciprocal-multiply adds 2 u.  With
    Q_i 2.2 |x_i| <= 0.81 that is Q_i (e^{2T} - 1 + (6 + 2 C) u) + u, first order, with 1 % for the rest."""
    return 1.01 * (np.asarray(q_ref) * (np.expm1(2 * T) + (6 + 2 * C) * U32) + U32)


def meanfield_exponent_bound(U, ys, weights, lats, dq_in=0.0, gains=None):
    """T: how far the exponent -U + sum_k w_k y_k of one mean-field step can be from fp64's when both start from the same Q
    (or from Q one dq_in apart, with gains[k] = max norm.K(norm.1)).  Each message y_k = norm.K(norm.Q) carries
    (L_k + 3 d_k + 7) u relative error: filter_rel_bound plus the weight products (the generic slice's w_k product, or the
    fast slice's three products folding alpha, norm and w_k into the weights).  Adding the messages to -U rounds once per
    lattice vertex gathered in the fast path's FMA chain (sum_k (d_k + 1), more than the generic path's one addition per
    kernel), each by at most u (|U| + sum_k w_k |y_k|)."""
    finite = np.isfinite(U)
    umax = float(np.abs(U[finite]).max()) if finite.any() else 0.0
    T, mag = 0.0, umax
    for k, (w, y, lat) in enumerate(zip(weights, ys, lats)):
        d = lat["offset"].shape[1] - 1
        ymax = float(np.nanmax(np.abs(y)))
        T += w * ymax * (max_row(lat) + 3 * d + 7) * U32
        if dq_in:
            T += w * gains[k] * dq_in
        mag += w * ymax
    return T + sum(lat["offset"].shape[1] for lat in lats) * U32 * mag


def unary_abs_bound(vmax, C):
    """pnp_crf_unary_from_maps against unary64, absolute: (x - min)/(max - min) is three roundings, at most 3 u vmax (vmax
    = max |v| of the row); v - max adds u 2 vmax, so every exponent is off by at most 8 u vmax; exp, the C - 1 additions of
    the sum and the division add (C + 3) u to log p; logf adds 1 ulp of |U| <= 11.6.  So 16 u vmax + (C + 3) u + 2 u 11.6."""
    return (16 * vmax + C + 3 + 24) * U32


# ----------------------------------------------------------------------------------------------- against the restatement
@pytest.fixture(scope="module")
def D():
    from oracle import densecrf
    try:
        densecrf.lib()
    except Exception as exc:  # noqa: BLE001 -- no C compiler: the restatement cannot be built here
        pytest.skip("oracle restatement not built: %s" % exc)
    return densecrf


def features(H, W, sxy, rgb=None, srgb=None):
    yy, xx = np.mgrid[0:H, 0:W]
    f = [xx.astype(np.float32) / np.float32(sxy), yy.astype(np.float32) / np.float32(sxy)]
    if rgb is not None:
        for c in range(3):
            f.append(rgb[:, :, c].astype(np.float32) / np.float32(srgb))
    return np.stack(f, -1).reshape(H * W, -1).astype(np.float32)


def oracle_lattice_arrays(ref, norm=None):
    """The restatement's lattice in the GPU's layout (nbr vertex + 1, 0 = none)."""
    nbr = np.stack([np.where(ref.n1 < 0, 0, ref.n1 + 1), np.where(ref.n2 < 0, 0, ref.n2 + 1)], -1)
    return dict(offset=ref.offset, bary=ref.barycentric, nbr=nbr, M=ref.M, norm=norm, shared=False)


H0, W0 = 37, 53


@pytest.mark.parametrize("kind", ["spatial", "bilateral"])
def test_filter64_is_the_unnormalised_restatement(D, kind):
    img = synth.guide_image(5, H0, W0)
    ref = D.Lattice(features(H0, W0, 3.0) if kind == "spatial" else features(H0, W0, 50.0, img, 5.0))
    lat = oracle_lattice_arrays(ref)
    x = np.random.default_rng(1).random((H0 * W0, 6)).astype(np.float32)
    want = splat_blur_slice64(lat, x)
    rel = float((np.abs(ref.compute(x) - want) / want).max())
    bound = filter_rel_bound(max_row(lat), lat["offset"].shape[1] - 1, normalized=False)
    print("%s: fp64 filter vs restatement, max relative error %.3g (bound %.3g)" % (kind, rel, bound))
    assert rel <= bound


def test_norm_kernel_apply_and_one_step_match_the_restatement(D):
    C = 7
    img = synth.guide_image(6, H0, W0)
    crf = D.DenseCRF2D(W0, H0, C)
    crf.addPairwiseGaussian(3, 7)
    crf.addPairwiseBilateral(50, 5, img, 10)
    lats = []
    for k, f in enumerate((features(H0, W0, 3.0), features(H0, W0, 50.0, img, 5.0))):
        lat = oracle_lattice_arrays(D.Lattice(f), crf.kernel_norm(k))
        d = lat["offset"].shape[1] - 1
        k1 = splat_blur_slice64(lat, np.ones((H0 * W0, 1)))[:, 0]
        norm64 = 1.0 / np.sqrt(k1 + 1e-20)
        rel = float(np.abs(lat["norm"] / norm64 - 1).max())
        assert rel <= filter_rel_bound(max_row(lat), d, False) / 2 + U32, (k, rel)
        x = np.random.default_rng(k).random((C, H0 * W0)).astype(np.float32)
        want = filter64(lat, x.T[None])[0].T
        rel = float((np.abs(crf.kernel_apply(k, x) - want) / want).max())
        bound = filter_rel_bound(max_row(lat), d, True)
        print("kernel %d: fp64 norm.K(norm.x) vs restatement, max relative error %.3g (bound %.3g)" % (k, rel, bound))
        assert rel <= bound
        lats.append(lat)
    # softmax64 and meanfield_step64 against DenseCRF2D.inference(0) and (1)
    rng = np.random.default_rng(3)
    p = rng.random((C, H0 * W0)).astype(np.float32) ** 3
    p /= p.sum(0, keepdims=True)
    Ucn = D.unary_from_softmax(p)
    crf.setUnaryEnergy(np.ascontiguousarray(Ucn))
    U = Ucn.T[None].astype(np.float64)
    q0 = softmax64(-U)
    b0 = softmax_bound(q0, C)
    assert (np.abs(crf.inference(0).T[None] - q0) <= b0).all()
    q1 = meanfield_step64(U, q0, lats, [7.0, 10.0])
    gains = [float(filter64(lat, np.ones((1, H0 * W0, 1))).max()) for lat in lats]
    T = meanfield_exponent_bound(U, messages64(q0, lats), [7.0, 10.0], lats, dq_in=float(b0.max()), gains=gains)
    err1 = np.abs(crf.inference(1).T[None] - q1)
    bound = softmax_bound(q1, C, T)
    print("one mean-field step: restatement vs fp64, max error %.3g, largest error / bound %.3g" % (err1.max(), (err1 / bound).max()))
    assert (err1 <= bound).all()


def test_unary64_matches_the_reference_formula(D):
    rng = np.random.default_rng(4)
    maps = (rng.random((2, 5, 300)) * 30).astype(np.float32)
    maps[1, 2, 17] = np.nan
    want = np.stack([D.unary_from_softmax(torch.softmax(torch.from_numpy(m).double(), 0).numpy()) for m in maps])
    got = unary64(maps)
    assert np.array_equal(np.isnan(got), np.isnan(np.moveaxis(want, 1, 2)))
    assert np.isnan(got[1, 17]).all() and not np.isnan(got[1, 16]).any()
    ok = ~np.isnan(got)
    assert np.abs(got[ok] - np.moveaxis(want, 1, 2)[ok]).max() <= 1e-6      # want is rounded to fp32
    assert (got[ok] == -np.log(1e-5)).any()                                   # the clip is reached


# ----------------------------------------------------------------------------------------------- the lattice shape limit
@pytest.fixture(scope="module")
def lib():
    from pnp_ovss_b200 import _lib
    try:
        return _lib.load()
    except (_lib.PnpError, OSError) as exc:
        pytest.skip("library not built: %s" % exc)


def table_capacity(d, n_pixels):
    cap = 1024
    while cap < 2 * n_pixels * (d + 1):
        cap <<= 1
    return cap


@pytest.mark.parametrize("d,side,limit", [(5, 512, 511), (5, 336, 1023), (2, 512, 1023)])
def test_lattice_slot_index_limit(lib, d, side, limit):
    """The build indexes every image's hash table with one int32 slot: n_images x capacity must stay <= INT32_MAX.  Init
    only carves pointers out of `storage`, so a dummy aligned address is enough to see where it refuses."""
    from pnp_ovss_b200 import _lib
    N = side * side
    assert limit * table_capacity(d, N) <= 2 ** 31 - 1 < (limit + 1) * table_capacity(d, N)
    assert (limit + 1) * N * (d + 1) < 0x7f000000                 # the entry-count limit is not what refuses
    for n, ok in ((limit, True), (limit + 1, False), (2 * limit, False)):
        lat = _lib.Lattice()
        rc = lib.pnp_lattice_init(ctypes.byref(lat), ctypes.c_void_p(1 << 20), 1 << 62, d, n, N, 0)
        assert rc == (PNP_OK if ok else PNP_ERR_INVALID_ARGUMENT), (d, side, n, rc)
        assert (lib.pnp_lattice_build_workspace_bytes(d, n, N) > 0) == ok
        assert (lib.pnp_lattice_storage_bytes(d, n, N) > 0) == ok
        if ok:
            assert lat.n_images == n and lat.vertex_stride == n * N * (d + 1)


def test_lattice_shape_limits(lib):
    from pnp_ovss_b200 import _lib
    lat = _lib.Lattice()
    big = ctypes.c_void_p(1 << 20)
    # one huge image: the entry-count limit (and no endless capacity loop past 2^31 slots)
    assert lib.pnp_lattice_init(ctypes.byref(lat), big, 1 << 62, 5, 1, 0x7f000000 // 6, 0) == PNP_ERR_INVALID_ARGUMENT
    assert lib.pnp_lattice_build_workspace_bytes(5, 1, 350_000_000) == 0
    assert lib.pnp_lattice_init(ctypes.byref(lat), big, 1 << 62, 5, 1, 4096 * 4096, 0) == PNP_OK
    assert lib.pnp_lattice_init(ctypes.byref(lat), big, 1 << 62, 2, 1, 336 * 336, 1) == PNP_OK
    assert lib.pnp_lattice_init(ctypes.byref(lat), big, 1 << 62, 2, 2, 336 * 336, 1) == PNP_ERR_INVALID_ARGUMENT
    assert lib.pnp_lattice_init(ctypes.byref(lat), ctypes.c_void_p((1 << 20) + 16), 1 << 62, 5, 1, 64, 0) == PNP_ERR_INVALID_ARGUMENT
