"""Small end-to-end cases shared by __graft_entry__.smoke() and the GPU tests: the CUDA pipeline and the CPU
oracle run the same seeded DRIVER_CASES inputs (tests/golden/make_golden_cases.py) and are compared."""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.dirname(HERE), os.path.join(HERE, "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import synth  # noqa: E402
from make_golden_cases import DRIVER_CASES, VOC_NMS  # noqa: E402


def case_inputs(tag):
    """Everything a DRIVER_CASES entry needs, loaded from the committed golden fixture."""
    g = np.load(os.path.join(HERE, "golden", "reference_golden.npz"), allow_pickle=False)
    coco, data_type, class_lists, R = DRIVER_CASES[tag]
    S, P, H, W, T, R_, n_cats = (int(v) for v in g["drv_%s_meta" % tag])
    tok = synth.SyntheticWordPieceTokenizer()
    caps = ["A picture of " + " ".join(cl) for cl in class_lists]
    tt = tok(caps, padding="max_length", max_length=500)
    if coco:
        catids = g["drv_%s_catids" % tag]
        ids = [[int(catids[VOC_NMS.index(c)]) for c in cl] for cl in class_lists]
        n_class = 91 if data_type == "coco_object" else 183
    else:
        ids = [[VOC_NMS.index(c) + 1 for c in cl] for cl in class_lists]
        n_class = n_cats + 1
    B = len(class_lists)   # the cases share one set of inputs; a case of B images takes the first B
    return dict(coco=coco, data_type=data_type, class_lists=class_lists, R=R, S=S, P=P, H=H, W=W, T=T, n_class=n_class,
                tok=tok, tokens=tt, rows=torch.from_numpy(g["drv_%s_rows" % tag]),
                imgs=torch.from_numpy(g["drv_imgs"][:B].copy()), gts=list(g["drv_gt"][:B]),
                guides=list(g["drv_guide"][:B]), ids=ids, golden=g)


def run_oracle(tag, mode):
    from oracle import hotpath as O
    c = case_inputs(tag)
    fn = synth.SynthGradcamFn(31, len(c["class_lists"]), c["T"], c["P"])
    with np.errstate(all="ignore"):
        h0, hagg, chosen = O.batch_confusion(lambda x: fn(x, c["rows"]), c["imgs"], c["tokens"].input_ids, c["tok"].decode,
                                             c["class_lists"], c["ids"], c["gts"], c["guides"], drop_iter=c["R"],
                                             patch_num=c["P"], threshold=0.15, data_type=c["data_type"], mode=mode,
                                             n_class=c["n_class"], coco=c["coco"], argsort_kind="stable")
    return h0, hagg


def run_gpu(tag, mode, dev):
    from pnp_ovss_b200 import pipeline
    c = case_inputs(tag)
    fn = synth.SynthGradcamFn(31, len(c["class_lists"]), c["T"], c["P"])
    h0, hagg, chosen = pipeline.batch_confusion(lambda x: fn(x.cpu(), c["rows"]).to(dev), c["imgs"].clone().to(dev),
                                                c["tokens"].input_ids.tolist(), c["tok"].decode, c["class_lists"], c["ids"],
                                                c["gts"], c["guides"], drop_iter=c["R"], patch_num=c["P"], threshold=0.15,
                                                data_type=c["data_type"], mode=mode, n_class=c["n_class"], coco=c["coco"])
    to_np = lambda h: None if h is None else h.cpu().numpy()
    return to_np(h0), to_np(hagg)


def disagreement(h_gpu, h_ref):
    """Fraction of pixels counted in a different (gt, pred) bin."""
    return float(np.abs(h_gpu.astype(np.float64) - h_ref).sum() / 2.0 / max(h_ref.sum(), 1.0))


def run_xattn(dev):
    """Rows a1/a2: the fused cross-attention softmax and softmax-backward/GradCAM kernels on the capture the reference's
    own code produced (golden gc_* vectors) and against the oracle's restatement."""
    from oracle import hotpath as O
    from pnp_ovss_b200 import ops
    g = np.load(os.path.join(HERE, "golden", "reference_golden.npz"), allow_pickle=False)
    probs = ops.softmax_fwd(torch.from_numpy(g["gc_scores_scaled"]).to(dev).contiguous(), None, 1.0)
    err = float(np.abs(probs.cpu().numpy() - g["gc_probs"]).max())
    assert err <= 1e-6, "softmax differs from the reference capture by %g" % err
    p, dp = torch.from_numpy(g["gc_probs"]), torch.from_numpy(g["gc_dprobs"])
    mask = torch.from_numpy(g["gc_mask500"])
    ds, cam = ops.softmax_bwd_gradcam(p.to(dev), dp.to(dev), mask.to(dev), 9, 0.125, True, True)
    want = g["gc_head9"]
    assert np.array_equal(cam.cpu().numpy().reshape(want.shape), want), "GradCAM differs from the reference's"
    ref_ds = O.softmax_backward(p, dp)
    assert np.allclose(ds.cpu().numpy(), ref_ds.numpy(), rtol=1e-4, atol=1e-9), "softmax backward differs from the oracle"
    return err


def run_model(dev):
    """A small BLIP-shaped model (head dimension 64) through the trimmed GradCAM pass in the shipped GEMM mode (3xFP16: fused
    operand kernels, the fp16x3 attention kernel, tensor-core text side, CUDA graphs) against torch's plain fp32 pass."""
    from pnp_ovss_b200.blip_itm import BlipITM
    tok = synth.SyntheticWordPieceTokenizer()
    caps = ["A picture of cat aeroplane", "A picture of dog"]
    tokens = tok(caps, padding="max_length", max_length=500).to(dev)
    torch.manual_seed(3)
    m = BlipITM(img_size=96, tokenizer=tok, hidden=128, layers=3, heads=2, inter=256, vit_dim=128, vit_depth=3, vit_heads=2, max_pos=64).eval()
    with torch.no_grad():
        for p_ in m.parameters():
            p_.mul_(2.0)
    m = m.to(dev).requires_grad_(False)
    imgs = torch.randn(2, 3, 96, 96, generator=torch.Generator().manual_seed(1)).to(dev)
    ref, _ = m.gradcam(imgs, caps, tokens, layer=1, head=1)
    m.gemm_precision = "3xfp16"
    got, _ = m.gradcam(imgs, caps, tokens, layer=1, head=1)
    again, _ = m.gradcam(imgs, caps, tokens, layer=1, head=1)         # second call: replayed from the captured graphs
    m.check_fp16_overflow()
    rel = float((got - ref).abs().max() / ref.abs().max())
    assert rel <= 1e-3 and torch.equal(got, again), "3xFP16 GradCAM differs from the fp32 pass by %g of its max" % rel
    return rel


def run(dev):
    """smoke(): the fused softmax/GradCAM kernels on the reference's capture, a small model pass in the shipped GEMM mode, then
    one DropOut + blur + CRF batch on the GPU against the oracle."""
    report = {"xattn_softmax_max_abs_err": run_xattn(dev), "model_3xfp16_vs_fp32_rel": run_model(dev)}
    for mode in ("blur", "blur+crf"):
        g0, gagg = run_gpu("voc_r4", mode, dev)
        o0, oagg = run_oracle("voc_r4", mode)
        assert g0.sum() == o0.sum() and gagg.sum() == oagg.sum(), "pixel totals differ"
        d0, dagg = disagreement(g0, o0), disagreement(gagg, oagg)
        report[mode] = (d0, dagg)
        limit = 0.0 if mode == "blur" else 0.01
        assert d0 <= limit and dagg <= limit, "GPU vs oracle pixel disagreement %g / %g in mode %s" % (d0, dagg, mode)
    return report
