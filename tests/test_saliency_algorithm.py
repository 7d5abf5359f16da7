"""The selection rule of pnp_salience_dropout_round and the summation order of pnp_token_merge, restated in numpy
(pnp_ovss_b200/csrc/gradcam.cu).  The GPU tests in test_gpu_saliency_contract.py hold the kernels to these restatements.

DropOut picks the save_len highest-scoring cells by rank counting: every cell p counts the cells q that rank above it and
writes itself to slot save_len-1-rank.  The reference takes np.argsort(score)[-save_len:]; the kernel matches the stable
sort.  The rank is a permutation -- each slot written exactly once -- only if the comparison is a total order.  A float
compare is not one once a score is NaN; the kernel compares order-preserving integer keys instead."""
import numpy as np
import pytest
import torch

from oracle import hotpath as O
from pnp_ovss_b200 import host

PPS = (441, 576, 784, 1024)     # P = 21, 24, 28, 32; 1024 is the kernel's kMaxCells
SAVE_LENS = (1, 10, 32)         # 32 is the largest save_len the kernel accepts


def score_key(s):
    """gradcam.cu score_key: float32 -> uint32, ascending in numpy's sort order (-0 == +0 < ... < +inf < NaN, NaNs equal)."""
    s = np.asarray(s, np.float32)
    u = np.where(s == 0, np.float32(0), s).astype(np.float32).view(np.uint32)
    key = np.where(u & np.uint32(0x80000000), ~u, u | np.uint32(0x80000000)).astype(np.uint32)
    return np.where(np.isnan(s), np.uint32(0xFFFFFFFF), key)


def _rank(greater, equal):
    """rank[p] = #(q ranks above p): greater[q, p] or (equal[q, p] and q > p)."""
    n = greater.shape[0]
    later = np.arange(n)[:, None] > np.arange(n)[None, :]
    return (greater | (equal & later)).sum(0)


def rank_float(s):
    """The parent kernel's rule: float compares, which are all false against NaN."""
    s = np.asarray(s, np.float32)
    return _rank(s[:, None] > s[None, :], s[:, None] == s[None, :])


def rank_key(s):
    """The kernel's rule: the same count over score_key."""
    k = score_key(s)
    return _rank(k[:, None] > k[None, :], k[:, None] == k[None, :])


def slot_writers(rank, save_len):
    """writers[j] = the cells that store themselves to s_new[j] (cell p writes slot save_len-1-rank[p] if rank[p] < save_len)."""
    writers = [[] for _ in range(save_len)]
    for p in np.flatnonzero(rank < save_len):
        writers[save_len - 1 - rank[p]].append(int(p))
    return writers


def select(s, save_len):
    """The cells the kernel writes to chosen[n_prev:n_prev+save_len], in slot order."""
    writers = slot_writers(rank_key(s), save_len)
    assert all(len(w) == 1 for w in writers)
    return np.array([w[0] for w in writers])


def _scores(kind, PP, rng):
    if kind == "random":
        return rng.standard_normal(PP).astype(np.float32)
    if kind == "tied":
        return rng.integers(0, 4, PP).astype(np.float32)
    if kind == "all_zero":
        return np.zeros(PP, np.float32)
    if kind == "signed_zero":
        s = np.where(rng.random(PP) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
        s[rng.choice(PP, 5, replace=False)] = rng.integers(-2, 3, 5)
        return s
    if kind == "inf":
        s = rng.integers(-3, 4, PP).astype(np.float32)
        s[rng.choice(PP, 40, replace=False)] = np.inf
        s[rng.choice(PP, 40, replace=False)] = -np.inf
        return s
    if kind == "some_nan":
        s = rng.integers(-3, 4, PP).astype(np.float32)
        s[rng.choice(PP, 5, replace=False)] = np.inf
        s[rng.choice(PP, 7, replace=False)] = np.nan
        return s
    if kind == "mostly_nan":
        s = np.full(PP, np.nan, np.float32)
        s[rng.choice(PP, 4, replace=False)] = rng.integers(-2, 3, 4)
        return s
    if kind == "all_nan":
        return np.full(PP, np.nan, np.float32)
    raise ValueError(kind)


KINDS = ("random", "tied", "all_zero", "signed_zero", "inf", "some_nan", "mostly_nan", "all_nan")


def test_score_key_orders_like_numpy():
    v = np.array([-np.inf, -3e38, -1.0, -1e-45, -0.0, 0.0, 1e-45, 1.0, 3e38, np.inf, np.nan], np.float32)
    k = score_key(v).astype(np.int64)
    assert (np.diff(k[[0, 1, 2, 3, 4, 6, 7, 8, 9, 10]]) > 0).all()
    assert k[4] == k[5]
    nans = np.array([np.nan, -np.nan], np.float32)
    nans = np.concatenate([nans, np.array([0x7FC00001, 0xFFFFFFFF], np.uint32).view(np.float32)])
    assert (score_key(nans) == 0xFFFFFFFF).all()


@pytest.mark.parametrize("PP", PPS)
@pytest.mark.parametrize("kind", KINDS)
def test_key_rank_is_a_permutation_equal_to_stable_argsort(PP, kind):
    """The integer-key rank is a bijection onto 0..PP-1 and the slot order is np.argsort(kind="stable")'s tail, in order."""
    rng = np.random.default_rng(PP + 17 * KINDS.index(kind))
    s = _scores(kind, PP, rng)
    r = rank_key(s)
    assert np.array_equal(np.sort(r), np.arange(PP))
    order = np.argsort(s, kind="stable")
    assert np.array_equal(r[order], np.arange(PP)[::-1])    # the cell sorted last ranks 0
    for save_len in SAVE_LENS:
        assert np.array_equal(select(s, save_len), order[-save_len:])


@pytest.mark.parametrize("PP", PPS)
def test_float_rank_agrees_with_key_rank_without_nan(PP):
    """Without NaN the two rules give the same ranks (only -0/+0 differ in key but never in float compare)."""
    rng = np.random.default_rng(PP)
    for kind in ("random", "tied", "all_zero", "signed_zero", "inf"):
        s = _scores(kind, PP, rng)
        assert np.array_equal(rank_float(s), rank_key(s)), kind


@pytest.mark.parametrize("PP", PPS)
def test_float_rank_is_not_a_permutation_with_nan(PP):
    """The float rule gives every NaN cell rank 0.  A few NaN cells: slot save_len-1 gets several writers (a race) and the
    other NaN cells are never chosen, while argsort would choose them first.  Fewer finite cells than save_len: slots stay
    unwritten, and the kernel would read uninitialised shared memory as cell indices."""
    rng = np.random.default_rng(PP)
    s = _scores("some_nan", PP, rng)
    writers = slot_writers(rank_float(s), 10)
    assert len(writers[9]) == 1 + int(np.isnan(s).sum())
    assert set(np.flatnonzero(np.isnan(s))) <= set(np.argsort(s, kind="stable")[-10:])
    for kind in ("mostly_nan", "all_nan"):
        s = _scores(kind, PP, rng)
        for save_len in SAVE_LENS[1:]:
            writers = slot_writers(rank_float(s), save_len)
            assert sum(len(w) == 0 for w in writers) == save_len - max(int(np.isfinite(s).sum()), 1), (kind, save_len)


# ------------------------------------------------------------------------------------------------ token merge
def token_merge_restated(g, seg_start, seg_len, seg_div, row_offset=3):
    """What pnp_token_merge computes, in float32: the first piece copied, the others added in token order (each sum rounded,
    __fadd_rn), one division (__fdiv_rn) when div != 1.  g [B,Tm,PP]; seg_* [B,C] -> [B,C,PP]."""
    g = np.asarray(g, np.float32)
    B, C = seg_start.shape
    out = np.zeros((B, C, g.shape[2]), np.float32)
    for b in range(B):
        for c in range(C):
            n = int(seg_len[b, c])
            if n == 0:
                continue
            rows = g[b, row_offset + int(seg_start[b, c]):]
            acc = rows[0].copy()
            for i in range(1, n):
                acc = acc + rows[i]
            d = np.float32(seg_div[b, c])
            out[b, c] = acc / d if d != 1 else acc
    return out


def wordpiece_tokens(pieces_per_word):
    """A caption's WordPiece strings after "a picture of": word w is "w<w>" followed by its "##p<k>" continuation pieces."""
    toks = []
    for w, n in enumerate(pieces_per_word):
        toks.append("w%d" % w)
        toks.extend("##p%d" % k for k in range(n - 1))
    return toks


def segment_tables(captions):
    """[(token strings, n_classes)] -> seg_start, seg_len int32 [B,Cmax], seg_div float32 [B,Cmax] via host.build_token_segments."""
    C = max(n for _, n in captions)
    start = np.zeros((len(captions), C), np.int32)
    length = np.zeros((len(captions), C), np.int32)
    div = np.ones((len(captions), C), np.float32)
    for b, (toks, n) in enumerate(captions):
        for c, (s, l, d) in enumerate(host.build_token_segments(toks, n)):
            start[b, c], length[b, c], div[b, c] = s, l, d
    return start, length, div


def test_token_merge_restatement_equals_the_reference_loop():
    """On random WordPiece captions (up to 171 words of up to 6 pieces), the restatement applied to host.build_token_segments'
    tables is bit-equal to the oracle's restatement of the reference loop (DRV:819-853)."""
    rng = np.random.default_rng(3)
    for trial in range(60):
        n_words = int(rng.choice([1, 2, 5, 9, 20, 150, 171])) if trial >= 10 else trial + 1
        pieces = rng.integers(1, 7 if trial % 2 else 3, n_words).tolist()
        toks = wordpiece_tokens(pieces)
        g = (rng.standard_normal((3 + len(toks) + 1, 4, 4)) * 10).astype(np.float32)
        start, length, div = segment_tables([(toks, n_words)])
        got = token_merge_restated(g.reshape(1, g.shape[0], 16), start, length, div)[0].reshape(n_words, 4, 4)
        want = O.mean_over_filtered_label_tokens(toks, torch.from_numpy(g), n_words).numpy()
        assert np.array_equal(got, want), pieces
