"""pnp_attention_fp16x3 at the edges of its arithmetic contract (pnp_ovss_b200/csrc/attention.cu), against an fp64 evaluation.

The kernel's softmax subtracts a per-row bound m_used that is refreshed -- and O, l rescaled in tensor memory -- only when the row
maximum grows by more than 2^8 (exp2 domain); the bound is the row maximum rounded up to bf16, exchanged by the two threads of a row;
P goes to the tensor cores as fp16 (hi, lo) pairs.  randn inputs almost never reach the rescale, nor the score magnitudes where the bf16
bound stops being exact.  These tests construct such inputs, check on the CPU restatement (test_attention_algorithm.py) that they reach
the path meant, and require the kernel to be as accurate as torch's own fp32 attention on the same input, or to raise its overflow
flag where the contract does not hold (the driver then repeats the run in 3xTF32)."""
import ctypes
import threading

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_attention_algorithm import (BOUND_LIMIT, SHIFTS_IN_RANGE, SHIFTS_PAST_BOUND, attention_tiled, expected_overflow_flag,
                                      shifted_head)

pytestmark = pytest.mark.gpu

LOG2E = 1.4426950408889634


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ops():
    from pnp_ovss_b200 import ops as _ops
    return _ops


def _sdpa(qkv, scale, dtype):
    B, L, _, H, D = qkv.shape
    q, k, v = (qkv[:, :, i].permute(0, 2, 1, 3).to(dtype) for i in range(3))
    return F.scaled_dot_product_attention(q, k, v, scale=scale).permute(0, 2, 1, 3).reshape(B, L, H * D)


def _run(ops, qkv, scale=0.125, in_scale=1.0, split_hi_scale=None):
    """(output, overflow flag) of one call."""
    flag = torch.zeros(1, dtype=torch.int32, device=qkv.device)
    out = ops.attention_fp16x3(qkv, in_scale=in_scale, softmax_scale=scale, flag=flag, split_hi_scale=split_hi_scale)
    return out, int(flag.item())


def _assert_fp32_grade(got, qkv, scale, in_scale=1.0):
    """max |got - fp64| / max |o| within 4x torch's fp32 SDPA error on the same input (+ 4e-6); NaN fails."""
    x = qkv.double() * in_scale
    truth = _sdpa(x, scale, torch.float64)
    sc = truth.abs().max().item()
    e_got = (got.double() - truth).abs().max().item() / sc
    e32 = (_sdpa(x.float(), scale, torch.float32).double() - truth).abs().max().item() / sc
    assert e_got <= 4 * e32 + 4e-6, "kernel %.3g, torch fp32 %.3g" % (e_got, e32)


def _stack(heads):
    """[(q, k, v) numpy [L, 64] per head] -> qkv [1, L, 3, H, 64] fp32 on the CPU."""
    return torch.from_numpy(np.stack([np.stack(h, 1) for h in heads], 2)[None].astype(np.float32))


def _rescales(heads, scale):
    return [attention_tiled(q, k, v, scale)[2] for q, k, v in heads]


def _ramp_head(L, growth, seed, rows=slice(None), scale=0.125):
    """randn k, v and q / 4; key j gets growth * (j // 64) (exp2 domain) added to its score on the given rows: a row's maximum grows
    by about `growth` per key tile.  The smaller q keeps the random part of the scores (sd ~0.35) from hiding a tile's growth, also
    on a last tile that holds a single key."""
    rng = np.random.default_rng(seed)
    q, k, v = (rng.standard_normal((L, 64)).astype(np.float32) for _ in range(3))
    q *= 0.25
    q[:, 0] = 0.0
    q[rows, 0] = 1.0
    k[:, 0] = growth / (scale * LOG2E) * (np.arange(L) // 64)
    return q, k, v


def _n_tiles(L):
    return (L + 63) // 64


# ------------------------------------------------------------------------------------------------ the lazy rescale
@pytest.mark.parametrize("L", [442, 1025])
def test_rescale_on_every_row_and_tile(dev, ops, L):
    """Every row's maximum grows by ~12 per tile: O in tensor memory and l are rescaled on every row at every tile after the first."""
    heads = [_ramp_head(L, 12.0, seed=L + h) for h in range(2)]
    assert _rescales(heads, 0.125) == [L * (_n_tiles(L) - 1)] * 2
    qkv = _stack(heads).to(dev)
    got, flag = _run(ops, qkv)
    _assert_fp32_grade(got, qkv, 0.125)
    assert flag == 0


def test_rescale_on_even_rows_only(dev, ops):
    """The ramp on even rows only: alpha = 1 lanes next to rescaled lanes of the same warp (the warp-divergent rescale)."""
    L = 442
    heads = [_ramp_head(L, 12.0, seed=7 + h, rows=slice(0, None, 2)) for h in range(2)]
    assert _rescales(heads, 0.125) == [(L + 1) // 2 * (_n_tiles(L) - 1)] * 2
    qkv = _stack(heads).to(dev)
    got, flag = _run(ops, qkv)
    _assert_fp32_grade(got, qkv, 0.125)
    assert flag == 0


def test_row_maximum_in_either_half_of_the_tile(dev, ops):
    """Even rows have each tile's maximum in keys 32-63, odd rows in keys 0-31, ~10 above the other half: the two threads of a row
    hold very different partial maxima and must still subtract the same bound and take the same rescale decision."""
    L, scale = 442, 0.125
    heads = []
    for h in range(2):
        q, k, v = _ramp_head(L, 12.0, seed=11 + h)
        a = 5.0 / (scale * LOG2E)
        k[:, 1] = np.where(np.arange(L) % 64 >= 32, a, -a)
        q[:, 1] = np.where(np.arange(L) % 2 == 0, 1.0, -1.0)
        heads.append((q, k, v))
    assert _rescales(heads, scale) == [L * (_n_tiles(L) - 1)] * 2
    qkv = _stack(heads).to(dev)
    got, flag = _run(ops, qkv, scale)
    _assert_fp32_grade(got, qkv, scale)
    assert flag == 0


def _threshold_head(L, tile_max, seed, scale=0.125):
    """Scores built from two dims only: key j's score is tile_max[j // 64] (exp2 domain) minus w_row * u_j, u_j in [0, 1.5] and 0 on
    the first key of each tile, so each tile's row maximum is tile_max exactly (up to the rounding of the products)."""
    rng = np.random.default_rng(seed)
    q = np.zeros((L, 64), np.float32)
    k = rng.standard_normal((L, 64)).astype(np.float32)
    v = rng.standard_normal((L, 64)).astype(np.float32)
    q[:, 0] = 1.0
    q[:, 1] = rng.uniform(0.25, 1.0, L)
    k[:, 0] = np.asarray(tile_max, np.float64)[np.arange(L) // 64] / (scale * LOG2E)
    u = rng.uniform(0.0, 1.5, L)
    u[::64] = 0.0
    k[:, 1] = -u / (scale * LOG2E)
    return q, k, v


def test_maximum_growth_just_under_the_threshold(dev, ops):
    """Tile 0's maximum is -3.95, every later tile's +3.95: a growth of 7.9 never triggers the rescale, so p reaches ~2^7.9 and l
    grows by a few hundred per tile -- the largest values the fp16 (hi, lo) pairs of P have to hold."""
    L = 442
    heads = [_threshold_head(L, [-3.95] + [3.95] * (_n_tiles(L) - 1), seed=21 + h) for h in range(2)]
    for q, k, v in heads:
        _, p_max, rescales, _ = attention_tiled(q, k, v, 0.125)
        assert rescales == 0 and 2.0 ** 7.8 < p_max <= 256.0
    qkv = _stack(heads).to(dev)
    got, flag = _run(ops, qkv)
    _assert_fp32_grade(got, qkv, 0.125)
    assert flag == 0


def test_maximum_growth_just_over_the_threshold(dev, ops):
    """Tile maxima -12.15, -4.05, 4.05, 12.15: a growth of 8.1 rescales every row at every tile (magnitudes below 16 keep the bf16
    round-up of the bound under 0.1)."""
    L = 250
    heads = [_threshold_head(L, [-12.15, -4.05, 4.05, 12.15], seed=31 + h) for h in range(2)]
    assert _rescales(heads, 0.125) == [L * 3] * 2
    qkv = _stack(heads).to(dev)
    got, flag = _run(ops, qkv)
    _assert_fp32_grade(got, qkv, 0.125)
    assert flag == 0


# ------------------------------------------------------------------------------------------------ score magnitudes and the flag
@pytest.mark.parametrize("c", SHIFTS_IN_RANGE + SHIFTS_PAST_BOUND)
def test_common_shift_of_every_score(dev, ops, c):
    """Every score moved by exactly c (natural units).  A softmax does not change; the kernel stays fp32-grade while the bound is
    below 2^11 in the exp2 domain (|c| <= 1400) and raises the flag past it, where the bf16 bound loses the row's largest p."""
    heads = [shifted_head(c, L=442, seed=h) for h in range(2)]
    expected = any(expected_overflow_flag(q, k, v, 0.125) for q, k, v in heads)
    assert expected == (abs(c) * LOG2E >= BOUND_LIMIT)
    qkv = _stack(heads).to(dev)
    got, flag = _run(ops, qkv)
    assert flag == int(expected)
    if not expected:
        _assert_fp32_grade(got, qkv, 0.125)
    assert _run(ops, qkv, split_hi_scale=1.0)[1] == int(expected)


@pytest.mark.parametrize("case", ["none", "q", "k", "v", "q_row_nan", "key_nan", "out3"])
def test_overflow_flag_per_operand_and_output_mode(dev, ops, case):
    """Each operand alone out of fp16's range after its scaling, or NaN, raises the flag in both output modes; an in-range input
    whose fp16 output split overflows (large split_hi_scale) raises it in the split mode only."""
    g = torch.Generator().manual_seed(5)
    qkv = torch.randn(2, 130, 3, 2, 64, generator=g)
    hi = 2.0
    if case == "q":
        qkv[1, 77, 0, 1, 5] = 4e5            # x 0.125 log2(e) = 72 000 > 65504
    elif case == "k":
        qkv[1, 77, 1, 1, 5] = 7e4
    elif case == "v":
        qkv[1, 77, 2, 1, 5] = 7e4
    elif case == "q_row_nan":
        qkv[0, 3, 0, 0, :] = float("nan")
    elif case == "key_nan":
        qkv[0, 100, 1, 1, 7] = float("nan")
    elif case == "out3":
        hi = 2.0 ** 20
    qkv = qkv.to(dev)
    assert _run(ops, qkv)[1] == int(case not in ("none", "out3")), "out"
    assert _run(ops, qkv, split_hi_scale=hi)[1] == int(case != "none"), "out3"


# ------------------------------------------------------------------------------------------------ workspace, layout, scales
def _abi_attention(lib, qkv, workspace, scale=0.125):
    B, L, _, H, D = qkv.shape
    out = torch.full((B, L, H * D), float("nan"), device=qkv.device)
    flag = torch.zeros(1, dtype=torch.int32, device=qkv.device)
    rc = lib.pnp_attention_fp16x3(ctypes.c_void_p(qkv.data_ptr()), 1.0, scale, ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(0), 1.0,
                                  ctypes.c_void_p(workspace.data_ptr()), workspace.numel(), ctypes.c_void_p(flag.data_ptr()), B, L, H, D,
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0
    return out, int(flag.item())


@pytest.mark.parametrize("L", [1, 65, 442, 1000])
def test_poisoned_workspace_does_not_leak(dev, L):
    """A workspace full of 0xFF bytes (fp16 NaN) gives the same output, bit for bit, as a zeroed one: the split pass writes every
    padded key row past L, so no 0 * NaN reaches P V."""
    from pnp_ovss_b200 import _lib
    lib = _lib.load()
    B, H = 2, 3
    qkv = torch.randn(B, L, 3, H, 64, generator=torch.Generator().manual_seed(L)).to(dev)
    ws = torch.empty(lib.pnp_attention_fp16x3_workspace_bytes(B, L, H, 64), dtype=torch.uint8, device=dev)
    clean, f0 = _abi_attention(lib, qkv, ws.zero_())
    poisoned, f1 = _abi_attention(lib, qkv, ws.fill_(0xFF))
    assert torch.equal(clean, poisoned) and f0 == 0 and f1 == 0
    _assert_fp32_grade(clean, qkv, 0.125)


def test_every_head_is_computed_alone(dev, ops):
    """B = 3, H = 16, each head at its own scale: every (b, h) output is bit-identical to a run of that head alone, so no batch,
    head or q/k/v stride mixes heads up (a single comparison with fp64 could average such an error away)."""
    B, L, H = 3, 200, 16
    g = torch.Generator().manual_seed(3)
    head_scale = (0.25 + 0.25 * torch.arange(H, dtype=torch.float32)).view(1, 1, 1, H, 1)
    qkv = (torch.randn(B, L, 3, H, 64, generator=g) * head_scale).to(dev)
    got, flag = _run(ops, qkv)
    assert flag == 0
    _assert_fp32_grade(got, qkv, 0.125)
    for b in range(B):
        for h in range(H):
            alone, _ = _run(ops, qkv[b:b + 1, :, :, h:h + 1].contiguous())
            assert torch.equal(got[b, :, 64 * h:64 * (h + 1)], alone[0]), (b, h)


@pytest.mark.parametrize("in_scale", [2.0 ** -11, 2.0 ** -3, 2.0 ** 4])
def test_in_scale_is_exact(dev, ops, in_scale):
    """qkv stored times 1/in_scale (a power of two) gives the in_scale = 1 output bit for bit, in both output modes."""
    qkv = torch.randn(2, 300, 3, 4, 64, generator=torch.Generator().manual_seed(9)).to(dev)
    for hi in (None, 2.0):
        ref, f0 = _run(ops, qkv, split_hi_scale=hi)
        got, f1 = _run(ops, (qkv / in_scale).contiguous(), in_scale=in_scale, split_hi_scale=hi)
        assert torch.equal(got, ref) and f0 == 0 and f1 == 0


@pytest.mark.parametrize("scale", [1.0, 0.05])
def test_softmax_scale(dev, ops, scale):
    """softmax_scale other than 1/sqrt(64): 1.0 spreads randn scores eight times wider (frequent rescales), 0.05 flattens them."""
    qkv = torch.randn(2, 442, 3, 4, 64, generator=torch.Generator().manual_seed(13)).to(dev)
    got, flag = _run(ops, qkv, scale)
    _assert_fp32_grade(got, qkv, scale)
    assert flag == 0


# ------------------------------------------------------------------------------------------------ production shapes, concurrency
@pytest.mark.parametrize("B,L,H", [(35, 442, 16), (35, 785, 16), (1, 2049, 4)])
def test_production_shapes(dev, ops, B, L, H):
    """configs[1] (442 tokens) and configs[4] (785) at 35 images x 16 heads, and 2049 keys (33 tiles: many mbarrier phases, an odd
    tile count): fp32-grade and deterministic."""
    qkv = torch.randn(B, L, 3, H, 64, generator=torch.Generator().manual_seed(L)).to(dev)
    got, flag = _run(ops, qkv)
    again, _ = _run(ops, qkv)
    assert flag == 0 and torch.equal(got, again)
    _assert_fp32_grade(got, qkv, 0.125)


def test_concurrent_calls_on_two_streams(dev, ops):
    """Two host threads, each on its own stream, call the attention at the same time (the header allows it): each result equals
    the serial call's bit for bit."""
    g = torch.Generator().manual_seed(1)
    inputs = [torch.randn(4, 442, 3, 16, 64, generator=g).to(dev), torch.randn(2, 785, 3, 16, 64, generator=g).to(dev)]
    serial = [ops.attention_fp16x3(x) for x in inputs]
    torch.cuda.synchronize(dev)
    reps = 4
    results = [[None] * reps for _ in inputs]
    errors = []
    barrier = threading.Barrier(len(inputs))

    def work(i):
        try:
            stream = torch.cuda.Stream(device=dev)
            with torch.cuda.stream(stream):
                barrier.wait()
                for r in range(reps):
                    results[i][r] = ops.attention_fp16x3(inputs[i])
            stream.synchronize()
        except BaseException as e:  # noqa: BLE001 -- reported by the main thread
            errors.append(e)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(inputs))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    for i, x in enumerate(inputs):
        for r in range(reps):
            assert torch.equal(results[i][r], serial[i]), (i, r)
