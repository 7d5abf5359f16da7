"""CPU: pin the oracle (oracle/hotpath.py) against outputs of the REFERENCE's own functions
(tests/golden/reference_golden.npz, produced by tests/golden/make_golden.py)."""
import numpy as np
import torch

import synth
from make_golden_cases import DRIVER_CASES, MERGE_CASES, VOC_NMS
from oracle import hotpath as O


def test_scale_0_1(golden):
    out = O.scale_0_1(torch.from_numpy(golden["scale01_in"].copy()))
    assert np.array_equal(out.numpy(), golden["scale01_out"])


def test_fast_hist_and_scores(golden):
    n = int(golden["hist_n"])
    gt, pred = golden["hist_gt"], golden["hist_pred"]
    assert np.array_equal(O.fast_hist(gt.flatten(), pred.flatten(), n), golden["hist_out"])
    table, hist = O.scores([gt, gt.T.copy()], [pred, pred.T.copy()], n)
    assert np.array_equal(hist, golden["scores_hist"])
    assert table["Mean IoU"] == float(golden["scores_miou"])
    assert table["Pixel Accuracy"] == float(golden["scores_acc"])
    assert table["Frequency Weighted IoU"] == float(golden["scores_fwiou"])


def test_blurring(golden):
    for tag in ("a", "b"):
        x = golden["blur_%s_in" % tag]
        y = O.blurring(torch.from_numpy(x), x.shape, scale=0.05)
        assert np.array_equal(y, golden["blur_%s_out" % tag])
    x = np.random.default_rng(int(golden["blur_c_in_seed"])).random((336, 336)).astype(np.float32)
    y = O.blurring(torch.from_numpy(x), (336, 336))
    assert np.array_equal(y[::16, ::16], golden["blur_c_out_sub"])


def test_token_merge(golden):
    tok = synth.SyntheticWordPieceTokenizer()
    for name, class_lists in MERGE_CASES.items():
        for cl in class_lists:  # register pieces in the same order as the generator
            tok("A picture of " + " ".join(cl))
    for name, class_lists in MERGE_CASES.items():
        ids = golden["merge_%s_ids" % name]
        g = torch.from_numpy(golden["merge_%s_g" % name])
        for b, cl in enumerate(class_lists):
            toks = O.token_strings(ids[b], tok.decode)
            out = O.mean_over_filtered_label_tokens(toks, g[b], len(cl))
            assert np.array_equal(out.numpy(), golden["merge_%s_out%d" % (name, b)]), (name, b)


def test_token_merge_split_last_is_summed_not_averaged(golden):
    """Quirk a3: a split word in LAST position is summed (DRV:844-847 divides only when a next token exists)."""
    g = torch.from_numpy(golden["merge_split_last_g"])
    out = golden["merge_split_last_out0"]  # classes [dog, aeroplane]; aeroplane = aero ##plan ##e
    rows = g[0][3:-1]
    assert np.allclose(out[1], (rows[1] + rows[2] + rows[3]).numpy())
    assert not np.allclose(out[1], ((rows[1] + rows[2] + rows[3]) / 3).numpy())


def test_gradcam_from_capture(golden):
    probs = torch.from_numpy(golden["gc_probs"])
    dprobs = torch.from_numpy(golden["gc_dprobs"])
    m500 = torch.from_numpy(golden["gc_mask500"])
    P = int(golden["gc_P"])
    assert np.array_equal(O.gradcam_head(probs, dprobs, m500, P, 9).numpy(), golden["gc_head9"])
    assert np.array_equal(O.gradcam_head(probs, dprobs, m500, P, 0).numpy(), golden["gc_head0"])
    # a1: the reference's nn.Softmax over the already-scaled scores
    s = torch.from_numpy(golden["gc_scores_scaled"])
    assert np.array_equal(O.cross_attention_probs(s * 2.0, None, head_size=4).numpy(), golden["gc_probs"])


def test_dropout_loop(golden):
    imgs = torch.from_numpy(golden["drop_imgs"])
    rows = torch.from_numpy(golden["drop_rows"])
    T = int(golden["drop_T"])
    B, P = imgs.shape[0], 6
    for R in (1, 4):
        fn = synth.SynthGradcamFn(21, B, T, P)
        g0, agg, chosen, _ = O.salience_dropout(lambda x: fn(x, rows), imgs, R, P)
        assert np.array_equal(g0.numpy(), golden["drop_R%d_g0" % R])
        if R > 1:
            assert np.array_equal(agg.numpy(), golden["drop_R%d_agg" % R])
            # quirk a4: the first round is counted twice
            assert not np.array_equal(agg.numpy(), golden["drop_R%d_g0" % R])
            assert all(len(c) == 10 * R for c in chosen)


def _run_driver_case(golden, tag, argsort_kind=None):
    coco, data_type, class_lists, R = DRIVER_CASES[tag]
    S, P, H, W, T, R_, n_cats = (int(v) for v in golden["drv_%s_meta" % tag])
    tok = synth.SyntheticWordPieceTokenizer()
    caps = ["A picture of " + " ".join(cl) for cl in class_lists]
    tt = tok(caps, padding="max_length", max_length=500)
    B = len(class_lists)   # the cases share one set of inputs; a case of B images takes the first B
    rows = torch.from_numpy(golden["drv_%s_rows" % tag])
    imgs = torch.from_numpy(golden["drv_imgs"][:B].copy())
    gts = list(golden["drv_gt"][:B])
    guides = list(golden["drv_guide"][:B])
    fn = synth.SynthGradcamFn(31, len(caps), T, P)
    if coco:  # sparse category ids (cats[idx]['id'], DRVC:549-584) and the COCO matrix sizes (DRVC:597-600)
        catids = golden["drv_%s_catids" % tag]
        ids = [[int(catids[VOC_NMS.index(c)]) for c in cl] for cl in class_lists]
        n_class = 91 if data_type == "coco_object" else 183
    else:
        ids = [[VOC_NMS.index(c) + 1 for c in cl] for cl in class_lists]
        n_class = n_cats + 1
    return O.batch_confusion(lambda x: fn(x, rows), imgs, tt.input_ids, tok.decode, class_lists, ids, gts, guides,
                             drop_iter=R, patch_num=P, threshold=0.15, data_type=data_type, mode="blur",
                             n_class=n_class, coco=coco, argsort_kind=argsort_kind)


def test_driver_end_to_end_hists(golden):
    """The reference's save_img_union_attention (real code, --postprocess blur) vs the oracle composition."""
    for tag in DRIVER_CASES:
        with np.errstate(all="ignore"):   # 0/0 channels are reference behaviour (DRV:1151-1152)
            h0, hagg, _ = _run_driver_case(golden, tag)
        k0, kagg = "drv_%s_hist_withfiltered_caption" % tag, "drv_%s_all_drop_hist_with_filtered_caption" % tag
        if h0 is not None:
            assert np.array_equal(h0, golden[k0]), tag
        if h0 is None:  # the COCO driver skips the round-0 pass when drop_iter >= 3 (DRVC:420, 602)
            assert k0 not in golden.files
        if hagg is not None:
            assert np.array_equal(hagg, golden[kagg]), tag
        else:
            assert kagg not in golden.files


def test_relabel_aliasing_quirk():
    """a9: classes [bicycle(2), aeroplane(1)]: local 2 -> id 1+... sequential rewrite aliases."""
    m = np.array([[0, 1, 2]], dtype=np.float32)
    # dataset ids for local classes: local1 -> 2, local2 -> 1 ; loop runs i=1 (local 2 -> 1) then i=0 (local 1 -> 2):
    # the pixel just written to 1 is rewritten to 2.
    out = O.relabel_sequential(m.copy(), [2, 1], with_background=True)
    assert out.tolist() == [[0, 2, 2]]
