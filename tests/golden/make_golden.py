#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REFERENCE's own functions (read from /root/reference at
generation time, in the build container only) on the seeded inputs of tests/golden/synth.py.

The reference module cannot be imported whole (lavis, pydensecrf, ... are absent), so the needed function /
class definitions are lifted out of the reference files with `ast` and exec'd unmodified in a namespace that
provides their imports.  Nothing is copied into the repo: only the OUTPUT arrays are committed.

Stubs (everything else is the reference's code):
  * the tokenizer (no bert vocab offline)          -> synth.SyntheticWordPieceTokenizer
  * dataset file loaders (no datasets)             -> synthetic GT / guide images
  * the BLIP model inside compute_gradcam_ensemble -> a tiny 12-layer stack built from the reference's OWN
    BertSelfAttention class (med.py:126-311) so capture + hook + autograd are the reference's
  * compute_gradcam_ensemble inside the DropOut-loop fixture -> synth.SynthGradcamFn
  * densecrf(): NOT exercised here (pydensecrf absent) -- fixtures use --postprocess blur; CRF is unpinned.

Run:  python tests/golden/make_golden.py      (needs /root/reference; the tests do not)
"""
import argparse
import ast
import math
import os
import sys
import types

import numpy as np
import torch
from torch import nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import synth  # noqa: E402

REF = "/root/reference"
DRV = os.path.join(REF, "PnP_OVSS_0514_updated_segmentation.py")
DRVC = os.path.join(REF, "PnP_OVSS_0514_updated_segmentation_coco.py")
BITM = os.path.join(REF, "Files to replace for BLIP", "blip_image_text_matching.py")
MED = os.path.join(REF, "Files to replace for BLIP", "med.py")


def lift(path, names, ns):
    """exec the named top-level defs of `path`, unmodified, into namespace ns."""
    src = open(path).read()
    tree = ast.parse(src)
    found = set()
    for node in tree.body:
        if isinstance(node, (ast.FunctionDef, ast.ClassDef)) and node.name in names:
            mod = ast.Module(body=[node], type_ignores=[])
            exec(compile(mod, path, "exec"), ns)
            found.add(node.name)
    missing = set(names) - found
    assert not missing, missing
    return ns


def base_ns():
    import json
    import time
    from pathlib import Path
    import torch.nn.functional as F
    from scipy.ndimage import filters
    return dict(torch=torch, np=np, nn=nn, math=math, F=F, filters=filters, json=json, time=time, Path=Path, os=os)


# --------------------------------------------------------------------------------------------------
def golden_small_functions(out):
    ns = lift(DRV, ["Scale_0_1", "_fast_hist", "scores", "blurring"], base_ns())
    rng = np.random.default_rng(11)
    # Scale_0_1 on a [C,H,W] map
    a = torch.from_numpy(rng.random((3, 9, 7)).astype(np.float32))
    out["scale01_in"] = a.numpy().copy()
    out["scale01_out"] = ns["Scale_0_1"](a.clone()).numpy()
    # _fast_hist with ignore label 255 and float32 gt
    n = 7
    gt = synth.gt_labels(5, 40, 36, n, ignore_frac=0.05, blocky=False)
    pred = rng.integers(0, n, (40, 36)).astype(np.float32)
    out["hist_gt"], out["hist_pred"], out["hist_n"] = gt, pred, np.int64(n)
    out["hist_out"] = ns["_fast_hist"](gt.flatten(), pred.flatten(), n)
    cats = {i: "c%d" % i for i in range(1, n)}
    table, hist = ns["scores"]([gt, gt.T.copy()], [pred, pred.T.copy()], cats, n)
    out["scores_hist"] = hist
    out["scores_miou"] = np.float64(table["Mean IoU"])
    out["scores_acc"] = np.float64(table["Pixel Accuracy"])
    out["scores_fwiou"] = np.float64(table["Frequency Weighted IoU"])
    # blurring on odd sizes (reflect boundary, radius > size/2 cases too)
    for tag, (H, W) in {"a": (48, 40), "b": (21, 64)}.items():
        x = rng.random((H, W)).astype(np.float32)
        x[x < 0.5] = 0
        out["blur_%s_in" % tag] = x
        out["blur_%s_out" % tag] = ns["blurring"](torch.from_numpy(x), (H, W), scale=0.05)
    x = rng.random((336, 336)).astype(np.float32)
    out["blur_c_in_seed"] = np.int64(77)
    x = np.random.default_rng(77).random((336, 336)).astype(np.float32)
    y = ns["blurring"](torch.from_numpy(x), (336, 336), scale=0.05)
    out["blur_c_out_sub"] = y[::16, ::16].copy()  # subsample keeps the fixture small


# --------------------------------------------------------------------------------------------------
def golden_token_merge(out):
    ns = lift(DRV, ["Mean_over_filtered_label_tokens"], base_ns())
    tok = synth.SyntheticWordPieceTokenizer()
    model = types.SimpleNamespace(module=types.SimpleNamespace(tokenizer=tok))
    cases = MERGE_CASES
    P = 5
    for name, class_lists in cases.items():
        caps = ["A picture of " + " ".join(c) for c in class_lists]
        tt = tok(caps, padding="max_length", max_length=500)
        T = int(tt.attention_mask.sum(1).max())
        g = torch.Generator().manual_seed(hash(name) % 1000 if False else len(name))
        grad = torch.rand(len(caps), T - 1, P, P, generator=g)
        grad = grad * tt.attention_mask[:, 1:T].view(len(caps), T - 1, 1, 1)
        out["merge_%s_ids" % name] = tt.input_ids[:, :T].numpy()
        out["merge_%s_g" % name] = grad.numpy()
        for b in range(len(caps)):
            r = ns["Mean_over_filtered_label_tokens"](model, tt, grad[b], class_lists, b)
            out["merge_%s_out%d" % (name, b)] = r.numpy().copy()
    out["merge_cases"] = np.array(sorted(cases))
    return cases


# --------------------------------------------------------------------------------------------------
class TinyCrossStack(nn.Module):
    """12 layers of the reference's BertSelfAttention used as cross-attention, wired with the attribute path
    compute_gradcam_ensemble walks (BITM:390-392)."""

    def __init__(self, SelfAttn, tok, P, enc_width=32, hidden=48, heads=12):
        super().__init__()
        cfg = types.SimpleNamespace(hidden_size=hidden, num_attention_heads=heads, encoder_width=enc_width,
                                    attention_probs_dropout_prob=0.0)
        self.tokenizer = tok
        self.P = P
        self.embed = nn.Embedding(31000, hidden)
        self.patch = nn.Linear(3 * 16 * 16, enc_width)
        layers = []
        for _ in range(12):
            layer = nn.Module()
            layer.crossattention = nn.Module()
            layer.crossattention.self = SelfAttn(cfg, True)
            layer.out = nn.Linear(hidden, hidden)
            layers.append(layer)
        enc = nn.Module()
        enc.layer = nn.ModuleList(layers)
        inner = nn.Module()
        inner.encoder = enc
        inner.base_model = inner
        self.text_encoder = nn.Module()
        self.text_encoder.base_model = inner
        self.head = nn.Linear(hidden, 2)
        self.captured_scores = {}

    def forward(self, samples, match_head="itm"):
        image, caption = samples["image"], samples["text_input"]
        B, _, S, _ = image.shape
        P = S // 16
        patches = image.reshape(B, 3, P, 16, P, 16).permute(0, 2, 4, 1, 3, 5).reshape(B, P * P, 768)
        emb = self.patch(patches)
        emb = torch.cat([emb.mean(1, keepdim=True), emb], 1)  # a CLS-like key in column 0
        text = self.tokenizer(caption, padding="longest")
        h = self.embed(text.input_ids)
        for i, layer in enumerate(self.text_encoder.base_model.encoder.layer):
            ctx = layer.crossattention.self(h, encoder_hidden_states=emb, encoder_attention_mask=None)[0]
            h = h + torch.tanh(layer.out(ctx))
        return self.head(h[:, 0, :])


def golden_gradcam(out):
    ns = base_ns()
    lift(MED, ["BertSelfAttention"], ns)
    lift(BITM, ["compute_gradcam_ensemble"], ns)
    torch.manual_seed(3)
    tok = synth.SyntheticWordPieceTokenizer()
    S, P = 96, 6
    model = TinyCrossStack(ns["BertSelfAttention"], tok, P)
    for p in model.parameters():
        torch.nn.init.normal_(p, 0, 0.3)
    caps = ["A picture of cat aeroplane", "A picture of dog"]
    imgs = torch.randn(2, 3, S, S)
    tt = tok(caps, padding="max_length", max_length=500)
    args = types.SimpleNamespace(img_size=S)
    # record the raw scores of block 7 on the way: wrap the reference softmax input via a forward pre-hook on
    # the module is not possible (scores are internal), so recompute them below from Q,K.
    blocklist, cam_list, itm = ns["compute_gradcam_ensemble"](args, model, imgs, caps, tt)
    att = model.text_encoder.base_model.base_model.encoder.layer[7].crossattention.self
    out["gc_probs"] = att.get_attention_map().detach().numpy()
    out["gc_dprobs"] = att.get_attn_gradients().detach().numpy()
    out["gc_mask500"] = tt.attention_mask.numpy()
    out["gc_P"] = np.int64(P)
    out["gc_head9"] = blocklist[7][9].numpy()
    out["gc_head0"] = blocklist[7][0].numpy()
    out["gc_itm"] = itm.detach().numpy()
    assert cam_list == []
    # scores -> probs pair for the softmax kernel: the reference's own module, hooked at nn.Softmax
    captured = {}
    orig = nn.Softmax.forward

    def spy(self_, x):
        captured.setdefault("scores", []).append(x.detach().clone())
        return orig(self_, x)
    nn.Softmax.forward = spy
    try:
        model({"image": imgs, "text_input": caps})
    finally:
        nn.Softmax.forward = orig
    out["gc_scores_scaled"] = captured["scores"][7].numpy()  # = QK^T / sqrt(head_size), MED:267


# --------------------------------------------------------------------------------------------------
def golden_dropout_loop(out):
    ns = lift(DRV, ["Inference_BLIP_filteredcaption"], base_ns())
    tok = synth.SyntheticWordPieceTokenizer()
    S, P, B = 96, 6, 3
    caps = ["A picture of cat aeroplane", "A picture of dog", "A picture of bus car person"]
    tt = tok(caps, padding="max_length", max_length=500)
    T = int(tt.attention_mask.sum(1).max())
    rows = tt.attention_mask[:, 1:T].float()
    imgs = torch.randn(B, 3, S, S, generator=torch.Generator().manual_seed(9))
    norm_imgs = imgs.permute(0, 2, 3, 1).contiguous().clone()
    for R in (1, 4):
        fn = synth.SynthGradcamFn(21, B, T, P)

        def fake_cge(args, model, visual_input, text_input, tokenized_text, drop_iter=0):
            g = fn(visual_input, rows)
            return [[g for _ in range(12)] for _ in range(12)], [], None
        ns["compute_gradcam_ensemble"] = fake_cge
        args = types.SimpleNamespace(drop_iter=R, img_size=S, max_att_block_num=8, prune_att_head=9,
                                     del_patch_num="sort_thresh005")
        model = types.SimpleNamespace(module=types.SimpleNamespace(tokenizer=tok))
        g0, agg = ns["Inference_BLIP_filteredcaption"](args, model, tt, imgs.clone(), norm_imgs.clone(),
                                                       ["11", "12", "13"], caps,
                                                       [c.split()[3:] for c in caps], "cpu")
        out["drop_R%d_g0" % R] = g0.numpy()
        if agg is not None:
            out["drop_R%d_agg" % R] = agg.numpy()
    out["drop_imgs"] = imgs.numpy()
    out["drop_rows"] = rows.numpy()
    out["drop_T"] = np.int64(T)


# --------------------------------------------------------------------------------------------------
def golden_driver(out, drv_path, tag, data_type, class_lists, nms, drop_iter, n_cats):
    """Run the reference's save_img_union_attention end to end (blur only) and capture the saved hists."""
    names = ["save_img_union_attention", "Inference_BLIP_filteredcaption", "Mean_over_filtered_label_tokens", "postprocess",
             "blurring", "Scale_0_1", "_fast_hist", "scores"]
    if drv_path == DRVC:
        names.append("getClassName")  # the COCO twin's scores() labels its table through it (DRVC:1315, 1355)
    ns = lift(drv_path, names, base_ns())
    tok = synth.SyntheticWordPieceTokenizer()
    S, P = 96, 6
    B = len(class_lists)
    H, W = 50, 44
    img_ids = [str(100 + i) for i in range(B)]
    gts = [synth.gt_labels(40 + i, H, W, n_cats + 1, ignore_frac=0.03) for i in range(B)]
    guides = [synth.guide_image(60 + i, H, W) for i in range(B)]
    best_idx = [[nms.index(c) for c in cl] for cl in class_lists]
    caps = ["A picture of " + " ".join(cl) for cl in class_lists]
    tt = tok(caps, padding="max_length", max_length=500)
    T = int(tt.attention_mask.sum(1).max())
    rows = tt.attention_mask[:, 1:T].float()
    fn = synth.SynthGradcamFn(31, B, T, P)

    def fake_cge(args, model, visual_input, text_input, tokenized_text, drop_iter=0):
        g = fn(visual_input, rows)
        return [[g for _ in range(12)] for _ in range(12)], [], None

    def fake_lpc(args, nms_, *rest, pred_path=None):
        if drv_path == DRVC:  # the COCO twin passes `cats` first (DRVC:858)
            rest = rest[1:]
        bl, cl, capl, gtl, ids, img = rest[:6]
        bl.append(list(best_idx[img]))
        cl.append(list(class_lists[img]))
        capl.append(caps[img])
        return bl, cl, capl

    saved = {}

    class NP:  # numpy with save() captured
        def __getattr__(self, k):
            return getattr(np, k)

        def save(self, path, arr):
            saved[os.path.basename(os.path.dirname(path))] = np.array(arr)

    ns.update(compute_gradcam_ensemble=fake_cge, Load_predicted_classes=fake_lpc,
              load_OrgImage=lambda a, ids, *ct: guides, Load_GroundTruth=lambda a, ids, *ct: gts, np=NP(),
              Draw_Segmentation_map=lambda *a, **k: None,
              # the COCO twin dumps JPEG overlays unconditionally (DRVC:829-844): visualisation stubs, no arithmetic
              getAttMap=lambda img, att, blur=True: np.zeros((2, 2, 3)),
              Image=types.SimpleNamespace(fromarray=lambda *a, **k: types.SimpleNamespace(save=lambda *a, **k: None)))
    # Path(...).mkdir writes under /tmp
    layers = [types.SimpleNamespace(crossattention=types.SimpleNamespace(self=types.SimpleNamespace(save_attention=True)))
              for _ in range(12)]
    inner = types.SimpleNamespace(encoder=types.SimpleNamespace(layer=layers))
    inner.base_model = inner
    module = types.SimpleNamespace(tokenizer=tok, text_encoder=types.SimpleNamespace(base_model=inner))
    model = types.SimpleNamespace(module=module)
    args = types.SimpleNamespace(drop_iter=drop_iter, img_size=S, max_att_block_num=8, prune_att_head=9,
                                 del_patch_num="sort_thresh005", threshold=0.15, data_type=data_type,
                                 postprocess="blur", save_path="/tmp/pnp_golden_%s" % tag, in_the_wild=False)
    imgs = torch.randn(B, 3, S, S, generator=torch.Generator().manual_seed(19))
    norm_imgs = imgs.permute(0, 2, 3, 1).contiguous().clone()
    if drv_path == DRVC:
        cats = {i: {"id": 3 * i + 1, "name": n} for i, n in enumerate(nms)}  # sparse ids like COCO
    else:
        cats = {i + 1: n for i, n in enumerate(nms)}
    lead = (None,) if drv_path == DRVC else ()  # DRVC:338 takes the pycocotools handle first
    ns["save_img_union_attention"](*lead, model, imgs, None, args, None, img_ids, drop_iter, norm_imgs, None, cats, nms,
                                   tt, "cpu", 9, max_block_num=8)
    for k, v in saved.items():
        out["drv_%s_%s" % (tag, k)] = v
    # every case draws its images, ground truth and guides from the same seeds: stored once, as long as the largest batch,
    # and a case of B images reads the first B (keeps the fixture under 1 MB)
    for k, v in (("imgs", imgs.numpy()), ("gt", np.stack(gts)), ("guide", np.stack(guides))):
        short, long_ = sorted((out.get("drv_" + k, v), v), key=len)
        assert np.array_equal(long_[:len(short)], short), k
        out["drv_" + k] = long_
    out["drv_%s_rows" % tag] = rows.numpy()
    out["drv_%s_meta" % tag] = np.array([S, P, H, W, T, drop_iter, n_cats], dtype=np.int64)
    if drv_path == DRVC:
        out["drv_%s_catids" % tag] = np.array([cats[i]["id"] for i in range(len(nms))], dtype=np.int64)
    return saved


from make_golden_cases import DRIVER_CASES as _CASES, MERGE_CASES, VOC_NMS  # noqa: E402

DRIVER_CASES = {k: ((DRVC if v[0] else DRV),) + tuple(v[1:]) for k, v in _CASES.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(HERE, "reference_golden.npz"))
    a = ap.parse_args()
    out = {}
    golden_small_functions(out)
    golden_token_merge(out)
    golden_gradcam(out)
    golden_dropout_loop(out)
    for tag, (drv, dt, cl, R) in DRIVER_CASES.items():
        golden_driver(out, drv, tag, dt, cl, VOC_NMS, R, len(VOC_NMS))
    np.savez_compressed(a.out, **out)
    print("wrote", a.out, "%.1f KB" % (os.path.getsize(a.out) / 1024), len(out), "arrays")


if __name__ == "__main__":
    main()
