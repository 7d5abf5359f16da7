"""CPU: the host side of segmenting images without ground truth -- the --in_the_wild flags, class-list parsing, output names,
the blur's size refusal, shard assignment and the whole driver loop (segment_images replaced by a stand-in), and
pipeline.batch_labels composed over shape-faithful stub ops (tests/stub_ops.py)."""
import argparse
import json
import os

import numpy as np
import pytest
import torch

import stub_ops
import synth
from pnp_ovss_b200 import driver, host, segment
from pnp_ovss_b200._lib import PnpError


def _parse(argv):
    return argparse.ArgumentParser(parents=[driver.get_args_parser()]).parse_args(argv)


def test_in_the_wild_flags_parse():
    a = _parse([])
    assert (a.in_the_wild, a.image_dir, a.classes, a.class_file) == (False, None, None, None)
    a = _parse("--in_the_wild --image_dir imgs --classes cat,dog --save_path out --img_size 336 --drop_iter 4 --threshold 0.15 "
               "--postprocess blur+crf --max_att_block_num 8 --prune_att_head 9 --gemm_precision 3xtf32".split())
    assert a.in_the_wild and (a.image_dir, a.classes, a.save_path, a.gemm_precision) == ("imgs", "cat,dog", "out", "3xtf32")


def test_class_names_from_classes_and_class_file(tmp_path):
    assert driver.parse_class_names(" cat, dog ,,grass ") == ["cat", "dog", "grass"]
    a = _parse(["--classes", "cat, potted plant"])
    assert driver.wild_class_lists(a, ["x", "y"]) == {"x": ["cat", "potted plant"], "y": ["cat", "potted plant"]}
    f = tmp_path / "map.json"
    f.write_text(json.dumps({"x": ["cat", " dog "], "y": "sky,road", "unused": ["a"]}))
    a = _parse(["--class_file", str(f)])
    assert driver.wild_class_lists(a, ["x", "y"]) == {"x": ["cat", "dog"], "y": ["sky", "road"]}
    with pytest.raises(SystemExit, match="no classes for z"):
        driver.wild_class_lists(a, ["x", "z"])
    for argv in ([], ["--classes", "cat", "--class_file", str(f)]):
        with pytest.raises(SystemExit, match="exactly one"):
            driver.wild_class_lists(_parse(argv), ["x"])
    with pytest.raises(SystemExit, match="1 to 255"):
        driver.wild_class_lists(_parse(["--classes", ",".join("c%d" % i for i in range(256))]), ["x"])
    with pytest.raises(SystemExit, match="1 to 255"):
        driver.wild_class_lists(_parse(["--classes", " , "]), ["x"])
    f.write_text(json.dumps([["cat"]]))
    with pytest.raises(SystemExit, match="JSON object"):
        driver.wild_class_lists(_parse(["--class_file", str(f)]), ["x"])
    # a multi-word name stays one word of the caption, so the token merge gives it one map
    assert segment.caption(["cat", "potted plant"]) == "A picture of cat pottedplant"


def test_image_listing_and_output_names(tmp_path):
    for name in ("b.PNG", "a.jpg", "c.jpeg", "notes.txt", "d.webp"):
        (tmp_path / name).write_bytes(b"")
    (tmp_path / "sub.png").mkdir()
    paths = driver.wild_images(str(tmp_path))
    assert list(paths) == ["a", "b", "c", "d"] and paths["b"] == os.path.join(str(tmp_path), "b.PNG")
    assert driver.wild_outputs("out", "a") == (os.path.join("out", "in_the_wild", "a.png"), os.path.join("out", "in_the_wild", "a_conf.npy"))
    (tmp_path / "a.png").write_bytes(b"")
    with pytest.raises(SystemExit, match="two images with the stem 'a'"):
        driver.wild_images(str(tmp_path))
    empty = tmp_path / "empty"
    empty.mkdir()
    with pytest.raises(SystemExit, match="no image"):
        driver.wild_images(str(empty))


def test_oversize_refusal_matches_the_blur_limit():
    from pnp_ovss_b200 import _lib
    lib = _lib.load()
    L = segment.BLUR_MAX_SIDE
    assert lib.pnp_gaussian_blur_workspace_bytes(1, 8, L, 0.05 * L) > 0
    assert lib.pnp_gaussian_blur_workspace_bytes(1, 8, L + 1, 0.05 * (L + 1)) == 0
    assert segment.size_refusal(L, 100, 2, "blur+crf") is None
    msg = segment.size_refusal(100, L + 1, 2, "blur+crf")
    assert msg and "1847 px" in msg and "100x1848" in msg
    assert segment.size_refusal(L + 1, 100, 2, "blur") is not None
    assert segment.size_refusal(L + 1, 100, 2, "crf") is None                       # no blur, no limit
    assert segment.size_refusal(L + 1, 100, 3, "blur+crf", "psc") is None           # no background channel
    # segment_images refuses before it touches the model or the GPU
    big = np.zeros((20, L + 1, 3), np.uint8)
    small = np.zeros((20, 30, 3), np.uint8)
    kw = dict(img_size=96, drop_iter=2, threshold=0.15, postprocess="blur+crf", max_att_block_num=2, prune_att_head=1)
    with pytest.raises(PnpError, match="image 1: .*1847 px"):
        segment.segment_images(None, [small, big], [["cat"], ["dog"]], **kw)
    with pytest.raises(PnpError, match="empty class list"):
        segment.segment_images(None, [small], [[]], **kw)
    with pytest.raises(PnpError, match="blank class name"):
        segment.segment_images(None, [small], [["cat", " "]], **kw)
    with pytest.raises(PnpError, match="2 images but 1 class lists"):
        segment.segment_images(None, [small, small], [["cat"]], **kw)


def test_load_model_image_takes_a_decoded_array_like_its_file(tmp_path):
    from PIL import Image
    from pnp_ovss_b200 import data
    rgb = synth.guide_image(3, 37, 52)
    Image.fromarray(rgb).save(tmp_path / "x.png")
    got = data.load_model_image(segment.load_rgb(str(tmp_path / "x.png")), 48)
    want = data.load_model_image(str(tmp_path / "x.png"), 48)
    assert torch.equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[2] == want[2] == (52, 37)
    assert np.array_equal(segment.load_rgb(rgb[..., 0]), np.stack([rgb[..., 0]] * 3, -1))
    with pytest.raises(PnpError):
        segment.load_rgb(rgb.astype(np.float32))


class _FakeModel:
    gemm_precision = "3xfp16"

    def __init__(self, overflow_once=False):
        self.flag = torch.tensor([1 if overflow_once else 0], dtype=torch.int32)

    def fp16_overflow_flag(self, dev):
        return self.flag


def _wild_tree(tmp_path):
    from PIL import Image
    d = tmp_path / "imgs"
    d.mkdir()
    sizes = {"a": (30, 40), "b": (44, 20), "c": (25, 25), "d": (12, 1900), "e": (33, 21)}
    for k, (H, W) in sizes.items():
        Image.fromarray(synth.guide_image(ord(k), H, W)).save(d / (k + (".jpg" if k == "b" else ".png")))
    return d, sizes


def test_driver_loop_shards_names_and_falls_back(tmp_path, monkeypatch, capsys):
    """main_in_the_wild with segment_images replaced by a stand-in: the oversize image is refused with its reason, the others
    are split into contiguous shards that together cover each image once, every rank writes its own files, rank 0 writes
    classes.json, and a raised fp16-range flag repeats the rank's images in 3xTF32."""
    from PIL import Image
    d, sizes = _wild_tree(tmp_path)
    calls = []

    def fake_segment_images(model, paths, class_lists, **kw):
        calls.append((model.gemm_precision, [os.path.basename(p) for p in paths], kw))
        out = []
        for p, c in zip(paths, class_lists):
            W, H = segment.image_size(p)
            ids = (np.arange(H * W).reshape(H, W) % (len(c) + 1)).astype(np.int32)
            out.append(dict(ids=ids, conf=np.full((H, W), 0.5, np.float32), classes=c))
        return out

    monkeypatch.setattr(segment, "segment_images", fake_segment_images)
    monkeypatch.setattr(torch.cuda, "set_device", lambda r: None)
    cls = tmp_path / "map.json"
    cls.write_text(json.dumps({"a": ["cat"], "b": ["cat", "dog"], "c": "sky,road,tree,car", "d": ["x"], "e": ["y", "z"]}))
    argv = ("--in_the_wild --image_dir %s --class_file %s --save_path %s --img_size 96 --batch_size 2 --drop_iter 2 --threshold 0.15 "
            "--postprocess blur+crf --max_att_block_num 2 --prune_att_head 1" % (d, cls, tmp_path / "out")).split()
    written = []
    for rank in range(3):
        written.append(driver.main_in_the_wild(rank, 3, _parse(argv), model=_FakeModel(overflow_once=rank == 1)))
    assert written == [["a", "b"], ["c"], ["e"]]
    assert [s for r in range(3) for s in ["a", "b", "c", "e"][slice(*host.shard_range(4, r, 3))]] == sum(written, [])
    assert "refused %s: image of 1900x12 px" % os.path.join(str(d), "d.png") in capsys.readouterr().out
    # rank 1 ran twice: 3xfp16, then 3xtf32 after its flag was raised
    assert [(c[0], c[1]) for c in calls] == [("3xfp16", ["a.png", "b.jpg"]), ("3xfp16", ["c.png"]), ("3xtf32", ["c.png"]),
                                             ("3xfp16", ["e.png"])]
    assert calls[0][2]["data_type"] == "voc" and calls[0][2]["postprocess"] == "blur+crf"
    out = tmp_path / "out" / "in_the_wild"
    assert json.loads((out / "classes.json").read_text()) == {"a": ["cat"], "b": ["cat", "dog"], "c": ["sky", "road", "tree", "car"],
                                                              "e": ["y", "z"]}
    assert sorted(os.listdir(out)) == ["a.png", "a_conf.npy", "b.png", "b_conf.npy", "c.png", "c_conf.npy", "classes.json", "e.png",
                                       "e_conf.npy"]
    for k, n_cls in (("a", 1), ("b", 2), ("c", 4), ("e", 2)):
        im = Image.open(out / (k + ".png"))
        H, W = sizes[k]
        assert im.mode == "P" and im.size == (W, H)
        assert np.array_equal(np.asarray(im), np.arange(H * W).reshape(H, W) % (n_cls + 1))
        assert np.load(out / (k + "_conf.npy")).shape == (H, W)


@pytest.fixture()
def pipe(monkeypatch):
    from pnp_ovss_b200 import ops, pipeline
    stub = stub_ops.make(ops)

    def label_map(labels, lut, Q=None):
        stub.calls.append("label_map")
        ok = (labels >= 0) & (labels < lut.shape[1])
        ids = torch.where(ok, torch.gather(lut.long(), 1, labels.long().clamp(0, lut.shape[1] - 1)), -1).to(torch.int32)
        conf = None if Q is None else torch.gather(Q, 2, labels.long().clamp(0, Q.shape[2] - 1)[..., None])[..., 0]
        return ids, conf

    stub.label_map = label_map
    monkeypatch.setattr(pipeline, "ops", stub)
    monkeypatch.setattr(pipeline, "_SPATIAL", pipeline.SpatialLatticeCache())
    pipeline._SEG_TABLES.clear()
    return pipeline, stub


@pytest.mark.parametrize("mode,drop_iter", [("blur+crf", 3), ("blur+crf", 1), ("blur", 2), ("", 2)])
def test_batch_labels_composes_ragged_batches_on_the_host(pipe, mode, drop_iter):
    """One post-processing pass per bucket (never a confusion matrix), maps at each image's guide size, in batch order."""
    pipeline, stub = pipe
    tok = synth.SyntheticWordPieceTokenizer()
    names = ["aeroplane", "bicycle", "bird", "boat"]
    class_lists = [names[:1], names[:2], names[:4], names[:1], names[:2]]
    shapes = [(30, 40), (30, 40), (24, 36), (24, 36), (20, 20)]
    caps = [segment.caption(c) for c in class_lists]
    tokens = tok(caps, padding="max_length", max_length=500)
    T = max(len(tok.encode(c)) for c in caps)
    S, P = 64, 4
    fn = synth.SynthGradcamFn(3, 5, T, P)
    rows = tokens.attention_mask[:, 1:T].float()
    guides = [synth.guide_image(20 + b, *shapes[b]) for b in range(5)]
    out = pipeline.batch_labels(lambda x: fn(x, rows), torch.randn(5, 3, S, S), tokens.input_ids.tolist(), tok.decode, class_lists, guides,
                                drop_iter=drop_iter, patch_num=P, threshold=0.15, data_type="voc", mode=mode)
    assert len(out) == 5
    for (ids, conf), c, hw in zip(out, class_lists, shapes):
        assert ids.dtype == torch.int32 and tuple(ids.shape) == hw
        assert int(ids.min()) >= 0 and int(ids.max()) <= len(c)
        assert (conf is None) == ("crf" not in mode) and (conf is None or tuple(conf.shape) == hw)
    n_buckets = len({(((len(c) + 1 + 3) // 4 * 4) if "blur" in mode else len(c), hw) for c, hw in zip(class_lists, shapes)})
    assert stub.calls.count("confusion_accumulate") == 0
    assert stub.calls.count("label_map") == n_buckets == stub.calls.count("lowrank_blur_unary" if "blur" in mode else "threshold_upsample")
    assert stub.calls.count("crf_inference") == (n_buckets if "crf" in mode else 0)
    assert stub.calls.count("token_merge") == 1                                 # one map per image: no separate round-0 pass
    assert stub.calls.count("salience_dropout_round") == (drop_iter if drop_iter > 1 else 0)
