"""The host planners of the post-processing kernels (pnp_ovss_b200/csrc/upsample_blur.cu, confusion.cu) restated in Python, and
the fp64 operators the GPU contract tests build their references from.  test_gpu_postprocess_contract.py takes its shapes and
its references from here.

The planners pick a kernel variant, a tiling and a loop structure from H and W alone, and real ground truths reach branches
that the benchmark's square shapes never do: two or more pass-H sweeps from 640 px wide, a second low-rank row chunk above 512
rows, the plain vertical kernel for an odd width, 16-row tiles from about 1.4k px, and refusal at 1847 px.  The restatement
names the branch of every shape; the tests below check that each GPU case reaches the branch it is meant to exercise and,
when the library is built, that the restatement accepts and sizes exactly what the library does (its *_workspace_bytes
entry points are host functions and run without a device)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

# ----------------------------------------------------------------------------------------------- constants of upsample_blur.cu
K_TAP_PAD, K_VCOLS, K_VROWS, K_TCOLS = 16, 64, 16, 32
K_HROWS, K_HCOLS, K_HGROUPS_MAX = 32, 16, 32
SMEM_BUDGET, TMA_BUDGET = 200 * 1024, 72 * 1024
K_LR_MAX_P = 32
LR_MAX_LW = (48 * 1024 - 128 * 8) // 16 - 1      # lowrank_operator_kernel: 2 lw + 1 doubles next to 1 KB, within 48 KB
BLUR_SCALE = 0.05                                # sigma = 0.05 * max(H, W) (DRV:1009)


def _align(x, a):
    return (x + a - 1) // a * a


def _cdiv(a, b):
    return -(-a // b)


def blur_radius(sigma):
    return int(4.0 * sigma + 0.5)                # scipy: int(truncate * sd + 0.5)


def blur_plan(n_maps, H, W, sigma, aligned=True):
    """make_blur_plan + the variant choices of blur_impl for maps [n_maps, H, W] at `aligned` (16-byte) input; None if refused."""
    if not sigma > 0 or n_maps < 0 or H < 1 or W < 1:
        return None
    lw = blur_radius(sigma)
    if lw > 4096:
        return None
    taps = 2 * lw + 1
    nwp = _align(taps, 8) + K_TAP_PAD
    fixed_rows = 2 * lw + K_TAP_PAD + K_VROWS
    max_rows = (SMEM_BUDGET - 4 * nwp) // (4 * K_VCOLS)
    if max_rows <= fixed_rows + K_VROWS:
        return None
    tile_rows = min(H, (max_rows - fixed_rows) // K_VROWS * K_VROWS)
    rows_max = (TMA_BUDGET - 4 * nwp) // (4 * K_TCOLS)
    tile_rows_tma = min(H, (rows_max - fixed_rows) // K_VROWS * K_VROWS) if rows_max > fixed_rows + K_VROWS else 0
    max_pitch = (SMEM_BUDGET - 4 * (nwp + K_HROWS * (K_HGROUPS_MAX * K_HCOLS + 1))) // (4 * K_HROWS)
    fixed_cols = 2 * lw + K_TAP_PAD + K_HCOLS
    if max_pitch <= fixed_cols + K_HCOLS + 1:
        return None
    tile_cols = min(W, (max_pitch - 1 - fixed_cols) // K_HCOLS * K_HCOLS)
    pitch = (tile_cols + fixed_cols) | 1
    n_col_groups = _cdiv(tile_cols, K_HCOLS)
    h_groups = _cdiv(n_col_groups, _cdiv(n_col_groups, K_HGROUPS_MAX))
    smem_h = 4 * (nwp + K_HROWS * pitch + K_HROWS * (h_groups * K_HCOLS + 1))
    tma = tile_rows_tma > 0 and W % 4 == 0 and aligned
    v_rows = tile_rows_tma if tma else tile_rows
    off_keys = _align(4 * nwp, 256)
    total = off_keys + _align(8 * n_maps, 256) + _align(4 * n_maps * H * W, 256)
    return dict(lw=lw, taps=taps, v="tma" if tma else "plain", v_rows=v_rows, v_tiles=_cdiv(H, v_rows),
                v_cols=K_TCOLS if tma else K_VCOLS, h_cols=tile_cols, h_tiles=_cdiv(W, tile_cols), h_groups=h_groups,
                h_sweeps=_cdiv(tile_cols, h_groups * K_HCOLS), h_pair=h_groups <= 21 and 2 * (smem_h + 1024) <= 227 * 1024,
                total=total)


def lowrank_plan(B, C, P, H, W, sigma, with_background):
    """make_lowrank_plan (after planning the background blur only when there is a background); None if refused."""
    if B < 0 or C < 1 or P < 1 or P > K_LR_MAX_P or H < 1 or W < 1 or not sigma > 0:
        return None
    blur = blur_plan(B, H, W, sigma) if with_background else None
    if with_background and blur is None:
        return None
    if not 4.0 * sigma + 0.5 < LR_MAX_LW + 1:
        return None
    ppad = 24 if P <= 24 else (28 if P <= 28 else 32)
    rows_chunk = min(H, 512)
    sweeps = _cdiv(W, 512)
    threads_a = min(512, max(64, _align(_cdiv(W, sweeps), 32)))
    cp = _align(C + (1 if with_background else 0), 4)
    tile_pix = 128 if cp <= 64 else 64
    smem_b = lambda tp: 4 * (C * ppad + 2 * C + tp * (cp + 1))   # noqa: E731
    if smem_b(tile_pix) > 200 * 1024:
        tile_pix = 32
        if smem_b(tile_pix) > 200 * 1024:
            return None
    bg = with_background
    sizes = [4 * B * C * P * P, 8 * B * C, 4 * H * ppad, 4 * W * ppad, 4 * B * C * H * ppad, 8 * B * C,
             4 * B * H * W if bg else 0, 4 * B * H * W if bg else 0, 8 * B if bg else 0, blur["total"] if bg else 0]
    return dict(ppad=ppad, row_chunks=_cdiv(H, rows_chunk), col_sweeps=_cdiv(W, threads_a), threads_a=threads_a,
                tile_pix=tile_pix, blur=blur, total=sum(_align(s, 256) for s in sizes))


def confusion_plan(N, n_class, aligned=True):
    """pnp_confusion_accumulate: vector or scalar items, and where the bins live."""
    smem = 4 * n_class * n_class
    bins = "smem" if smem <= 48 * 1024 else ("smem_optin" if smem <= 200 * 1024 else "global")
    return dict(vec=N % 4 == 0 and aligned, bins=bins)


def argmax_vec(N, aligned=True):
    return N % 4 == 0 and aligned


def upsample_vec(W, aligned=True):
    return W % 4 == 0 and aligned


# ----------------------------------------------------------------------------------------------- the GPU file's cases
# direct blur (one map, sigma = 0.05 max side, aligned input): the branch each shape is there for
BLUR_SHAPES = {
    (336, 336): dict(v="tma", v_tiles=1, h_pair=True, h_sweeps=1, h_tiles=1),
    (375, 500): dict(v="tma", v_tiles=2, h_pair=False, h_sweeps=1, h_tiles=1),
    (512, 512): dict(v="tma", v_tiles=2, h_pair=False, h_sweeps=1, h_tiles=1),
    (480, 640): dict(v="tma", h_sweeps=2, h_tiles=1),
    (427, 640): dict(v="tma", h_sweeps=2, h_tiles=1),
    (512, 683): dict(v="plain", v_tiles=2, h_sweeps=2, h_tiles=1),
    (683, 512): dict(v="tma", v_tiles=3, h_tiles=1),
    (513, 513): dict(v="plain", h_sweeps=2, h_tiles=1),
    (768, 1024): dict(h_tiles=2),
    (1024, 1365): dict(v="plain", v_tiles=5, h_tiles=3),
    (1380, 1847): dict(v="plain", v_rows=16, h_tiles=7),
    (1847, 1380): dict(v="plain", v_rows=16, v_tiles=116, h_tiles=5),
    (1847, 1847): dict(v="plain", v_rows=16, v_tiles=116, h_tiles=7),
}
# the plain-against-TMA comparison: the same maps through an input offset by one float
BLUR_PLAIN_VS_TMA = ((336, 336), (480, 640))
# fused low-rank group
LOWRANK_SHAPES = {
    (480, 640): dict(row_chunks=1, col_sweeps=2), (427, 640): dict(row_chunks=1, col_sweeps=2),
    (512, 683): dict(row_chunks=1, col_sweeps=2), (683, 512): dict(row_chunks=2, col_sweeps=1),
    (513, 513): dict(row_chunks=2, col_sweeps=2), (768, 1024): dict(row_chunks=2, col_sweeps=2),
    (1024, 1365): dict(row_chunks=2, col_sweeps=3), (1380, 1847): dict(row_chunks=3, col_sweeps=4),
}
LOWRANK_P = (21, 24, 25, 28, 32, 1)
LOWRANK_TINY = ((1, 97), (97, 1), (2, 2))
LOWRANK_WIDE_C = (171, 480, 640)       # C = 171 classes + background: tile_pix 64
LOWRANK_HUGE_C = (600, 64, 80)         # tile_pix 32
LOWRANK_NO_BG_LARGE = ((1848, 1848), (2400, 1800))   # past the direct blur's limit, fine without a background
# argmax / confusion: (B, H, W) at real ground-truth sizes
CONFUSION_SHAPES = ((35, 480, 640), (35, 375, 333), (35, 427, 641))
CONFUSION_N_CLASS = (21, 150, 171, 183, 300)
ARGMAX_C = (21, 151, 172)


@pytest.mark.parametrize("shape", sorted(BLUR_SHAPES))
def test_every_blur_case_reaches_its_branch(shape):
    H, W = shape
    p = blur_plan(1, H, W, BLUR_SCALE * max(H, W))
    assert p is not None
    for k, v in BLUR_SHAPES[shape].items():
        assert p[k] == v, (shape, k, p[k], v)


def test_the_blur_cases_cover_every_branch():
    plans = [blur_plan(1, H, W, BLUR_SCALE * max(H, W)) for H, W in BLUR_SHAPES]
    assert {p["v"] for p in plans} == {"tma", "plain"}
    assert {p["h_pair"] for p in plans} == {True, False}
    assert max(p["h_sweeps"] for p in plans) >= 2 and max(p["h_tiles"] for p in plans) >= 2
    assert any(p["v"] == "plain" and p["v_tiles"] >= 2 for p in plans) and any(p["v"] == "tma" and p["v_tiles"] >= 3 for p in plans)
    # the misaligned view forces the plain kernel where the aligned input takes the TMA one
    for H, W in BLUR_PLAIN_VS_TMA:
        s = BLUR_SCALE * max(H, W)
        assert blur_plan(1, H, W, s)["v"] == "tma" and blur_plan(1, H, W, s, aligned=False)["v"] == "plain"
    # 1024 x 1365: W % 4 != 0 is not why it is plain: the TMA tile no longer fits 72 KB at that sigma
    assert blur_plan(1, 1024, 1368, BLUR_SCALE * 1368)["v"] == "plain"


def test_the_limits_of_the_direct_blur():
    assert blur_plan(1, 1847, 1847, BLUR_SCALE * 1847) is not None
    assert blur_plan(1, 1848, 1848, BLUR_SCALE * 1848) is None
    assert blur_plan(1, 1848, 10, BLUR_SCALE * 1848) is None            # the radius decides, not the area
    assert blur_plan(1, 10, 10, 1024.2) is None and blur_radius(1024.2) > 4096


@pytest.mark.parametrize("shape", sorted(LOWRANK_SHAPES))
def test_every_lowrank_case_reaches_its_branch(shape):
    H, W = shape
    for bg in (0, 1):
        p = lowrank_plan(2, 5, 21, H, W, BLUR_SCALE * max(H, W), bg)
        for k, v in LOWRANK_SHAPES[shape].items():
            assert p[k] == v, (shape, bg, k, p[k], v)


def test_the_lowrank_cases_cover_every_template_and_tile():
    assert {lowrank_plan(1, 3, P, 64, 64, 3.2, 1)["ppad"] for P in LOWRANK_P} == {24, 28, 32}
    C, H, W = LOWRANK_WIDE_C
    assert lowrank_plan(1, C, 21, H, W, BLUR_SCALE * max(H, W), 1)["tile_pix"] == 64
    C, H, W = LOWRANK_HUGE_C
    assert lowrank_plan(1, C, 32, H, W, BLUR_SCALE * max(H, W), 1)["tile_pix"] == 32
    assert lowrank_plan(1, 3, 21, 64, 64, 3.2, 1)["tile_pix"] == 128
    for H, W in LOWRANK_NO_BG_LARGE:
        s = BLUR_SCALE * max(H, W)
        assert lowrank_plan(1, 3, 21, H, W, s, 0) is not None and lowrank_plan(1, 3, 21, H, W, s, 1) is None


def test_the_confusion_cases_cover_every_path():
    seen = set()
    for B, H, W in CONFUSION_SHAPES:
        for n in CONFUSION_N_CLASS:
            for aligned in (True, False):
                p = confusion_plan(H * W, n, aligned)
                seen.add((p["vec"], p["bins"]))
    assert seen == {(v, b) for v in (True, False) for b in ("smem", "smem_optin", "global")}
    assert not confusion_plan(375 * 333, 21)["vec"] and confusion_plan(480 * 640, 21)["vec"]
    assert {argmax_vec(H * W) for _, H, W in CONFUSION_SHAPES} == {True, False}


# ----------------------------------------------------------------------------------------------- against the library
@pytest.fixture(scope="module")
def lib():
    from pnp_ovss_b200 import _lib
    try:
        return _lib.load()
    except (_lib.PnpError, OSError) as exc:
        pytest.skip("library not built: %s" % exc)


def _boundary_grid():
    rng = np.random.default_rng(0)
    sides = [1, 2, 3, 97, 336, 500, 511, 512, 513, 640, 683, 1024, 1365, 1400, 1846, 1847, 1848, 1849, 2400, 4000]
    shapes = [(H, W) for H in sides for W in sides]
    shapes += [tuple(int(v) for v in rng.integers(1, 2600, 2)) for _ in range(300)]
    return shapes


def test_the_blur_boundary_equals_the_library(lib):
    for H, W in _boundary_grid():
        for sigma in (BLUR_SCALE * max(H, W), 0.7, 3.2):
            for n_maps in (1, 35):
                p = blur_plan(n_maps, H, W, sigma)
                assert lib.pnp_gaussian_blur_workspace_bytes(n_maps, H, W, sigma) == (p["total"] if p else 0), (n_maps, H, W, sigma)
    for sigma in (0.0, -1.0, 1023.8, 1024.2, 2000.0):
        p = blur_plan(1, 10, 10, sigma)
        assert lib.pnp_gaussian_blur_workspace_bytes(1, 10, 10, sigma) == (p["total"] if p else 0)
    assert lib.pnp_gaussian_blur_workspace_bytes(1, 10, 10, 1024.2) == 0          # radius 4097


def test_the_lowrank_boundary_equals_the_library(lib):
    for H, W in _boundary_grid():
        s = BLUR_SCALE * max(H, W)
        for B, C, P in ((1, 3, 21), (35, 20, 21), (2, 171, 28), (1, 600, 32), (1, 900, 32)):
            for bg in (0, 1):
                p = lowrank_plan(B, C, P, H, W, s, bg)
                got = lib.pnp_lowrank_blur_workspace_bytes(B, C, P, H, W, s, bg)
                assert got == (p["total"] if p else 0), (B, C, P, H, W, bg)
    # without a background the fused kernels' own limit applies: lowrank_operator_kernel's weights (lw <= 3007)
    for sigma, ok in ((751.8, True), (751.9, False)):
        assert (lib.pnp_lowrank_blur_workspace_bytes(1, 3, 21, 64, 64, sigma, 0) > 0) == ok
        assert (lowrank_plan(1, 3, 21, 64, 64, sigma, 0) is not None) == ok
    assert lib.pnp_lowrank_blur_workspace_bytes(1, 3, 21, 1848, 1848, BLUR_SCALE * 1848, 0) > 0
    assert lib.pnp_lowrank_blur_workspace_bytes(1, 3, 21, 1848, 1848, BLUR_SCALE * 1848, 1) == 0
    assert lib.pnp_lowrank_blur_workspace_bytes(1, 3, 33, 64, 64, 3.2, 0) == 0


# ----------------------------------------------------------------------------------------------- fp64 operators
def reflect_index(i, n):
    """scipy mode='reflect' (d c b a | a b c d | d c b a), vectorised."""
    i = np.asarray(i)
    if n == 1:
        return np.zeros_like(i)
    i = np.mod(i, 2 * n)
    return np.where(i < n, i, 2 * n - 1 - i)


def gauss_weights(sigma):
    """scipy's _gaussian_kernel1d(sigma, 0, int(4 sigma + 0.5)) in float64."""
    lw = blur_radius(sigma)
    x = np.arange(-lw, lw + 1, dtype=np.float64)
    w = np.exp(-0.5 / (sigma * sigma) * x * x)
    return w / w.sum()


def gauss_matrix(n, sigma):
    """G [n, n]: (G x)[y] = sum_j w[j] x[reflect(y + j - lw)], i.e. gaussian_filter1d(x, sigma, mode='reflect')."""
    w = gauss_weights(sigma)
    lw = (w.size - 1) // 2
    cols = reflect_index(np.arange(n)[:, None] + np.arange(-lw, lw + 1)[None, :], n)
    flat = (np.arange(n)[:, None] * n + cols).ravel()
    return np.bincount(flat, weights=np.tile(w, n), minlength=n * n).reshape(n, n)


def interp_matrix(n, P):
    """U [n, P]: bilinear, align_corners=True, from its formula: source s = y (P - 1) / (n - 1) (0 for n = 1)."""
    s = np.arange(n, dtype=np.float64) * ((P - 1) / (n - 1) if n > 1 else 0.0)
    i0 = np.minimum(np.floor(s).astype(np.int64), P - 1)
    i1 = np.minimum(i0 + 1, P - 1)
    lam = s - i0
    U = np.zeros((n, P))
    np.add.at(U, (np.arange(n), i0), 1.0 - lam)
    np.add.at(U, (np.arange(n), i1), lam)
    return U


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (2, 2), (2, 9), (7, 1), (13, 17), (40, 31)])
@pytest.mark.parametrize("sigma", [0.3, 0.7, 1.6, 4.0, 11.0])
def test_gauss_matrix_is_scipys_gaussian_filter(shape, sigma):
    from scipy.ndimage import gaussian_filter
    H, W = shape
    x = np.random.default_rng(H * 100 + W).standard_normal(shape)
    got = gauss_matrix(H, sigma) @ x @ gauss_matrix(W, sigma).T
    np.testing.assert_allclose(got, gaussian_filter(x, sigma), rtol=0, atol=1e-13)
    assert np.allclose(gauss_matrix(max(H, W), sigma).sum(1), 1.0, rtol=0, atol=1e-14)   # rows sum to one (the reflection folds)


@pytest.mark.parametrize("shape", [(1, 1), (1, 5), (2, 2), (2, 7), (5, 1), (31, 29), (336, 200)])
@pytest.mark.parametrize("P", [1, 2, 21, 32])
def test_interp_matrix_is_torch_bilinear_align_corners(shape, P):
    H, W = shape
    m = np.random.default_rng(P).standard_normal((P, P))
    want = F.interpolate(torch.from_numpy(m)[None, None], size=(H, W), mode="bilinear", align_corners=True)[0, 0].numpy()
    np.testing.assert_allclose(interp_matrix(H, P) @ m @ interp_matrix(W, P).T, want, rtol=0, atol=1e-13)

