"""GPU: segmenting images without ground truth.  pnp_label_map against numpy at its edges; pipeline.batch_labels on a ragged batch
(three sizes, 1 / 2 / 4 classes) against batch_confusion run on each image alone, bit for bit; the --in_the_wild driver end to
end against segment_images."""
import json
import os

import numpy as np
import pytest
import torch

import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def _label_map_ref(labels, lut, Q):
    B, N = labels.shape
    ids = np.full((B, N), -1, np.int32)
    conf = np.full((B, N), -1, np.float32)
    for b in range(B):
        ok = (labels[b] >= 0) & (labels[b] < lut.shape[1])
        ids[b, ok] = lut[b, labels[b, ok]]
        if Q is not None:
            conf[b, ok] = Q[b, np.nonzero(ok)[0], labels[b, ok]]
    return ids, conf


def _unaligned(t):
    """A contiguous copy of t whose data pointer is 4 bytes past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    out = buf[1:].view(t.shape)
    out.copy_(t)
    assert out.data_ptr() % 16 == 4
    return out


@pytest.mark.parametrize("B,N,Cp,lut_w", [(3, 1024, 4, 3), (2, 1001, 8, 5), (1, 4 * 37, 1024, 1000), (4, 333, 12, 12),
                                          (2, 48 * 40, 4, 2), (0, 64, 4, 3)])
@pytest.mark.parametrize("aligned", [True, False])
@pytest.mark.parametrize("with_q", [True, False])
def test_label_map_matches_numpy(dev, B, N, Cp, lut_w, aligned, with_q):
    from pnp_ovss_b200 import ops
    rng = np.random.default_rng(B * 7919 + N + Cp)
    labels = rng.integers(0, lut_w, size=(B, N)).astype(np.int32)
    if B:   # out of range on both sides, including the first label past the lut and past Q's channels
        labels[0, ::17] = -1
        labels[-1, 5::23] = lut_w
        labels[0, 3::29] = 2 ** 30
    lut = rng.integers(0, 200, size=(B, lut_w)).astype(np.int32)
    Q = rng.random((B, N, Cp)).astype(np.float32)
    if B:
        Q[0, 7] = np.nan       # a NaN row of Q: its marginal comes through as NaN
        Q[-1, N // 2, :] = np.nan
    Qd = torch.from_numpy(Q).to(dev) if with_q else None
    lab_d, lut_d = torch.from_numpy(labels).to(dev), torch.from_numpy(lut).to(dev)
    if not aligned and B:
        lab_d = _unaligned(lab_d)
    ids, conf = ops.label_map(lab_d, lut_d, Qd)
    if not aligned and B:   # and unaligned outputs, through the C ABI directly
        from pnp_ovss_b200 import _lib
        ids = _unaligned(torch.zeros_like(ids))
        conf = _unaligned(torch.zeros_like(conf)) if with_q else None
        _lib.check(_lib.load().pnp_label_map(ops._p(lab_d), ops._p(lut_d), lut_w, ops._p(Qd), Cp if with_q else 0, ops._p(ids), ops._p(conf),
                                             B, N, ops._stream()), "pnp_label_map")
    want_ids, want_conf = _label_map_ref(labels, lut, Q if with_q else None)
    assert ids.shape == (B, N) and np.array_equal(ids.cpu().numpy(), want_ids)
    if with_q:
        np.testing.assert_array_equal(conf.cpu().numpy(), want_conf)   # NaN where Q is NaN, -1 where the label is out of range
    else:
        assert conf is None


def test_label_map_refuses_bad_arguments(dev):
    from pnp_ovss_b200 import PnpError, _lib, ops
    lab = torch.zeros(2, 16, dtype=torch.int32, device=dev)
    lut = torch.zeros(2, 5, dtype=torch.int32, device=dev)
    with pytest.raises(PnpError):
        ops.label_map(lab, lut, torch.zeros(2, 16, 4, device=dev))      # Cp < lut columns: a label could read past Q
    with pytest.raises(PnpError):
        ops.label_map(lab, lut[:1])
    with pytest.raises(PnpError):
        ops.label_map(lab.float(), lut)
    lib = _lib.load()
    out = torch.empty_like(lab)
    q = torch.zeros(2, 16, 8, device=dev)
    assert lib.pnp_label_map(ops._p(lab), ops._p(lut), 5, ops._p(q), 8, ops._p(out), ops._p(None), 2, 16, ops._stream()) == -1
    assert lib.pnp_label_map(ops._p(lab), ops._p(lut), 5, ops._p(None), 0, ops._p(out), ops._p(q), 2, 16, ops._stream()) == -1


# ---------------------------------------------------------------------------------------------- ragged batch vs batches of one
def _tiny_model(tok, dev):
    from pnp_ovss_b200.blip_itm import BlipITM
    torch.manual_seed(11)
    m = BlipITM(img_size=96, tokenizer=tok, vocab=30524, hidden=128, layers=3, heads=2, inter=256, vit_dim=64, vit_depth=2,
                vit_heads=2, max_pos=64).eval()
    with torch.no_grad():   # as test_gpu_model_path: widen the random init so the maps have structure
        for p in m.parameters():
            p.mul_(2.0)
    return m.to(dev).requires_grad_(False)


NAMES = ["aeroplane", "bicycle", "bird", "boat", "motorbike"]
CLASS_LISTS = [NAMES[:1], NAMES[1:3], NAMES[:4], NAMES[2:3], NAMES[1:5]]
SHAPES = [(40, 56), (40, 56), (64, 48), (50, 50), (64, 48)]


@pytest.fixture(scope="module")
def ragged(dev):
    from pnp_ovss_b200 import segment
    tok = synth.SyntheticWordPieceTokenizer()
    model = _tiny_model(tok, dev)
    caps = [segment.caption(c) for c in CLASS_LISTS]
    tokens = [tok([c], padding="max_length", max_length=500).to(dev) for c in caps]
    Tm = max(len(tok.encode(c)) for c in caps) - 1

    def gradcam_fn(members):
        """Every image's map computed with the image alone and padded to the batch's row count: a batch and the batches of one
        of its images see the same maps and the same DropOut rows."""
        def fn(x):
            out = []
            for j, b in enumerate(members):
                g = model.gradcam(x[j:j + 1], [caps[b]], tokens[b], layer=1, head=1)[0]
                out.append(torch.cat([g, g.new_zeros((1, Tm - g.shape[1]) + tuple(g.shape[2:]))], 1))
            return torch.cat(out)
        return fn

    imgs = torch.randn(5, 3, 96, 96, generator=torch.Generator().manual_seed(5)).to(dev)
    guides = [synth.guide_image(40 + b, *SHAPES[b]) for b in range(5)]
    token_ids = [t.input_ids[0].tolist() for t in tokens]
    return dict(tok=tok, gradcam_fn=gradcam_fn, imgs=imgs, guides=guides, token_ids=token_ids)


@pytest.mark.parametrize("mode,drop_iter,key", [("blur+crf", 4, "all_drop"), ("blur+crf", 1, "round0"), ("blur", 4, "all_drop")])
@pytest.mark.parametrize("threads", [True, False])
def test_ragged_batch_labels_equal_batches_of_one(dev, ragged, monkeypatch, mode, drop_iter, key, threads):
    from pnp_ovss_b200 import ops, pipeline
    monkeypatch.setattr(pipeline, "BUCKET_THREADS", threads)
    kw = dict(drop_iter=drop_iter, patch_num=6, threshold=0.15, data_type="voc", mode=mode)
    got = pipeline.batch_labels(ragged["gradcam_fn"](range(5)), ragged["imgs"].clone(), ragged["token_ids"], ragged["tok"].decode,
                                CLASS_LISTS, ragged["guides"], **kw)
    torch.cuda.synchronize()
    seen = []
    crf_inference = ops.crf_inference

    def recording(lattices, weights, unary, C, n_iter, **k):
        Q, labels = crf_inference(lattices, weights, unary, C, n_iter, **k)
        seen.append((Q, C))
        return Q, labels

    monkeypatch.setattr(ops, "crf_inference", recording)
    for b in range(5):
        H, W = SHAPES[b]
        labels_out = {}
        seen.clear()
        h0, hall, _ = pipeline.batch_confusion(ragged["gradcam_fn"]([b]), ragged["imgs"][b:b + 1].clone(), ragged["token_ids"][b:b + 1],
                                               ragged["tok"].decode, [CLASS_LISTS[b]], [list(range(1, len(CLASS_LISTS[b]) + 1))],
                                               [np.full((H, W), -1, np.float32)], [ragged["guides"][b]], n_class=21, labels_out=labels_out, **kw)
        assert all(int(h.sum()) == 0 for h in (h0, hall) if h is not None)      # a ground truth of -1 counts nothing
        ids, conf = got[b]
        want = labels_out[key][0]
        assert ids.dtype == torch.int32 and ids.shape == (H, W)
        assert torch.equal(ids.float(), want), "image %d: %d pixels differ" % (b, int((ids.float() != want).sum()))
        assert 0 <= int(ids.min()) and int(ids.max()) <= len(CLASS_LISTS[b])
        if "crf" in mode:
            Q, C = seen[-1]                                         # the scored pass is the last CRF of the batch of one
            real = len(CLASS_LISTS[b]) + 1
            assert C == real and conf.shape == (H, W)
            assert torch.equal(conf, Q[0, :, :real].max(-1)[0].view(H, W))
        else:
            assert conf is None


# ---------------------------------------------------------------------------------------------- driver end to end
def test_in_the_wild_driver_end_to_end(dev, tmp_path, capsys):
    """PNG and JPEG images of mixed sizes, one past the blur's limit: the driver refuses that one with its reason and writes a
    palette PNG and a confidence map per other image that equal what segment_images gives for the same images.  The model is the
    tiny one above (a random-init full-size model's GradCAM on 96 px inputs is flat, and the reference's min-max turns flat maps
    into NaN)."""
    import argparse
    from PIL import Image
    from pnp_ovss_b200 import driver, segment_images
    d = tmp_path / "imgs"
    d.mkdir()
    sizes = {"cat_photo": (60, 80, ".jpg"), "street": (75, 50, ".png"), "field": (64, 64, ".jpeg"), "panorama": (24, 1900, ".png")}
    for k, (H, W, ext) in sizes.items():
        Image.fromarray(synth.guide_image(len(k), H, W)).save(d / (k + ext), quality=95)
    table = {"cat_photo": ["cat", "sofa"], "street": "car,person,road,building", "field": ["grass"], "panorama": ["sky"]}
    (tmp_path / "map.json").write_text(json.dumps(table))
    argv = ("--in_the_wild --image_dir %s --class_file %s --save_path %s --img_size 96 --batch_size 4 --max_att_block_num 2 "
            "--prune_att_head 1 --drop_iter 2 --threshold 0.15 --postprocess blur+crf --world_size 1 --gemm_precision fp32"
            % (d, tmp_path / "map.json", tmp_path / "out")).split()
    args = argparse.ArgumentParser(parents=[driver.get_args_parser()]).parse_args(argv)
    model = _tiny_model(synth.SyntheticWordPieceTokenizer(), dev)
    assert driver.main_in_the_wild(0, 1, args, model=model) == ["cat_photo", "field", "street"]
    log = capsys.readouterr().out
    assert "refused %s" % (d / "panorama.png") in log and "1847 px" in log
    out = tmp_path / "out" / "in_the_wild"
    classes = json.loads((out / "classes.json").read_text())
    assert sorted(os.listdir(out)) == sorted(["classes.json"] + [s + suf for s in classes for suf in (".png", "_conf.npy")])
    stems = sorted(classes)
    res = segment_images(model, [str(d / (s + sizes[s][2])) for s in stems], [classes[s] for s in stems], img_size=96, drop_iter=2,
                         threshold=0.15, postprocess="blur+crf", max_att_block_num=2, prune_att_head=1, batch_size=4)
    for s, r in zip(stems, res):
        H, W, _ = sizes[s]
        assert classes[s] == r["classes"] == (table[s].split(",") if isinstance(table[s], str) else table[s])
        im = Image.open(out / (s + ".png"))
        assert im.mode == "P" and im.size == (W, H)
        ids = np.asarray(im)
        assert ids.min() >= 0 and ids.max() <= len(classes[s])
        assert np.array_equal(ids, r["ids"])
        conf = np.load(out / (s + "_conf.npy"))
        assert conf.dtype == np.float32 and conf.shape == (H, W) and np.array_equal(conf, r["conf"])
        assert np.all((conf > 0) & (conf <= 1))
