"""Segmentation driver with the reference's CLI (PnP_OVSS_0514_updated_segmentation.py:57-106, 1193-1225, 1439):
same flag names and defaults, one process per GPU, data-parallel over images.

    python -m pnp_ovss_b200.driver --data_type voc --img_size 336 --batch_size 35 --max_att_block_num 8 \\
        --prune_att_head 9 --drop_iter 4 --del_patch_num sort_thresh005 --sort_threshold 0.05 --threshold 0.15 \\
        --postprocess blur+crf --world_size 1 --save_path out/

Differences from the reference, all forced by what exists offline:
  * the datasets, the GPT-4o class lists, the BLIP checkpoint and the bert vocabulary are absent, so images, ground
    truth, guide images, class lists and the tokenizer are the seeded stand-ins of pnp_ovss_b200.synthetic and the
    model is the random-init BlipITM of pnp_ovss_b200.blip_itm (`--synthetic_images N` sets the dataset size);
  * ranks take disjoint contiguous shards (host.shard_range) instead of DistributedSampler's padded shuffle, and the
    per-rank confusion matrices are summed with ONE int64 all-reduce over NCCL instead of through .npy files; rank 0
    still writes the matrix where Calculate_mIoU.py looks for it (DRV:513-520) and prints the same statistics.
`--sort_threshold` is accepted and unused, like in the reference (DRV:85-86 is never read).

With the real inputs on disk the same driver runs them (`main_real`):
    python -m pnp_ovss_b200.driver --real_data --home_dir /data --data_type voc --bert_vocab vocab.txt \\
        --checkpoint model_large_retrieval_flickr.pth --img_size 336 --batch_size 35 --max_att_block_num 8 ...
reads {home_dir}/VOCdevkit/VOC2012/{val.txt,JPEGImages,SegmentationClass} and {home_dir}/GPT4o_classification/*.json in the
reference's layouts (pnp_ovss_b200/data.py, reference_api.save_img_union_attention).

`--in_the_wild` segments your own images with class names you choose, without ground truth (segment.segment_images):
    python -m pnp_ovss_b200.driver --in_the_wild --image_dir photos/ --classes "cat,dog,grass" --save_path out/ \
        --img_size 336 --batch_size 35 --max_att_block_num 8 --prune_att_head 9 --drop_iter 4 --threshold 0.15 \
        --postprocess blur+crf [--bert_vocab vocab.txt --checkpoint model_large_retrieval_flickr.pth]
(`--class_file map.json` instead of --classes: a JSON object {image stem: [class names] or "a,b,c"}).  It writes
out/in_the_wild/<stem>.png (a palette PNG: 0 = background, i = the i-th class of the image), <stem>_conf.npy (float32, the CRF
marginal of each chosen label; modes with a CRF only) and classes.json ({stem: class list}).  Ranks take contiguous shards of
the images in name order and write their own files.  An image the blur cannot take is refused with the reason and skipped."""
import argparse
import json
import os
import time

import numpy as np
import torch

from . import data, host, pipeline, synthetic
from .reference_api import metrics_from_hist

DATASETS = {  # data_type -> (caption class names, n_class for the confusion matrix)   LD:8-92, DRV:496, DRVC:597-600
    "voc": (list(data.VOC_NAMES), 21),
    "psc": (list(data.CONTEXT_NAMES), 60),
    "ade20k": (["".join(n.split(" ")) for n in data.ADE_NAMES], 151),
    "coco_object": (["class%02d" % i for i in range(80)], 91),       # the COCO names live in the annotation file
    "coco_stuff": (["class%03d" % i for i in range(171)], 183),
}


def get_args_parser():
    """The reference's parser (DRV:57-106), flag for flag, plus the synthetic-data knobs."""
    parser = argparse.ArgumentParser('image caption localization with ITM', add_help=False)
    parser.add_argument('--batch_size', default=2, type=int)
    parser.add_argument('--num_workers', default=0, type=int)
    parser.add_argument('--gen_multiplecap_withpnpvqa', default="label")
    parser.add_argument('--save_path', default="Eval_test_ddp")
    parser.add_argument('--home_dir', default="/home/letitiabanana/LAVIS/")
    parser.add_argument('--master_port', default="12355")
    parser.add_argument('--existing_att_path', default="./Cbatch_Eval_test_ddp_0521_labelascaption/img_att_forclasses/")
    parser.add_argument("--cam_out_dir", default="./Eval_test_ddp_0331/img_att_forclasses/", type=str)
    parser.add_argument("--del_patch_num", default=None)
    parser.add_argument("--max_att_block_num", default=10, type=int)
    parser.add_argument("--img_size", default=768, type=int)
    parser.add_argument("--world_size", default=4, type=int)
    parser.add_argument("--ensemble_blocks", default=None, type=str)
    parser.add_argument("--drop_iter", default=10, type=int)
    parser.add_argument("--prune_att_head", default=None)
    parser.add_argument("--sort_threshold", default=None, type=float)
    parser.add_argument("--edge_map_for_clip", action="store_true")
    parser.add_argument("--final_att_threshold", default=0.05)
    parser.add_argument("--search", default=None)
    parser.add_argument("--layer", default=None, type=str)
    parser.add_argument("--cal_token_sim_forall_layerhead", action="store_true")
    parser.add_argument("--in_the_wild", action="store_true")
    parser.add_argument("--data_type", default=None, type=str)
    parser.add_argument("--postprocess", default=None, type=str)
    parser.add_argument("--threshold", default=None, type=float)
    # not in the reference: the data that replaces the absent datasets
    parser.add_argument("--synthetic_images", default=8, type=int, help="size of the synthetic dataset")
    parser.add_argument("--synthetic_classes", default=3, type=int, help="classes per image (captioned 'A picture of c1 c2 ...')")
    parser.add_argument("--synthetic_seed", default=1234, type=int)
    parser.add_argument("--real_data", action="store_true",
                        help="read images / ground truth / GPT-4o class lists from --home_dir in the reference's layouts "
                             "(needs --bert_vocab; --checkpoint for the real weights) instead of the synthetic stand-ins")
    parser.add_argument("--bert_vocab", default=None, type=str, help="local bert-base-uncased vocab.txt (the hub is offline)")
    parser.add_argument("--checkpoint", default=None, type=str, help="LAVIS BlipITM checkpoint (model_large_retrieval_flickr.pth)")
    parser.add_argument("--coco_annotation_file", default=None, type=str, help="instances_val2017.json (COCO category table)")
    parser.add_argument("--max_images", default=0, type=int, help="real data: evaluate only the first N images (0 = all)")
    parser.add_argument("--gemm_precision", default="3xfp16", choices=["fp32", "3xtf32", "3xfp16"],
                        help="how the model's dense contractions run: torch's native fp32 GEMMs, or fp32-grade error-compensated "
                             "products on the TF32 / fp16 tensor cores (the shipped default; DESIGN.md 3b).  A 3xfp16 run whose "
                             "activations leave fp16's range is repeated in 3xtf32.")
    parser.add_argument("--synthetic_gt_size", default=0, type=int,
                        help="side of the ground-truth / guide images (0 = img_size); the maps are upsampled to it (DRV:435-437)")
    parser.add_argument("--image_dir", default=None, type=str, help="--in_the_wild: the folder of images to segment")
    parser.add_argument("--classes", default=None, type=str, help="--in_the_wild: comma-separated class names for every image")
    parser.add_argument("--class_file", default=None, type=str,
                        help="--in_the_wild: JSON object {image stem: [class names] or 'a,b,c'} (instead of --classes)")
    return parser


def ddp_setup(args, rank, world_size):
    """DRV:45-54, with 127.0.0.1 instead of a hostname lookup."""
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", str(args.master_port))
    torch.distributed.init_process_group(backend="nccl", rank=rank, world_size=world_size)


def synthetic_shard(args, names, n_class, start, end):
    """Images [start, end) of the synthetic dataset (generated per image id, so shards do not depend on world_size)."""
    S = int(args.img_size)
    G = int(args.synthetic_gt_size) or S
    rng = np.random.default_rng(args.synthetic_seed)
    class_ids_all = [sorted(rng.choice(len(names), size=min(args.synthetic_classes, len(names)), replace=False).tolist())
                     for _ in range(args.synthetic_images)]
    items = []
    for i in range(start, end):
        g = torch.Generator().manual_seed(args.synthetic_seed + i)
        ids = class_ids_all[i]
        items.append(dict(img_id="syn_%06d" % i, img=torch.randn(3, S, S, generator=g), class_idx=ids,
                          classes=[names[c] for c in ids], gt=synthetic.gt_labels(args.synthetic_seed + i, G, G, n_class),
                          guide=synthetic.guide_image(args.synthetic_seed + i, G, G)))
    return items


def _fp16_range_exceeded(model, dev, world_size):
    """True on every rank when any rank's 3xFP16 operand kernels saw an activation outside fp16's range (the device flag is read
    here, once per run)."""
    if model.gemm_precision != "3xfp16":
        return False
    flag = model.fp16_overflow_flag(dev).clone()
    if world_size > 1:
        torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MAX)
    return bool(int(flag.item()))


def main_real(rank, world_size, args, model=None):
    """captions_text_loc (DRV:1090-1188) on the real directory layouts: images from disk through the reference's
    transform, then reference_api.save_img_union_attention per batch (which reads guide images, ground truth and GPT-4o
    class lists itself and writes the per-batch .npy matrices), the matrices summed on the device and all-reduced."""
    from . import reference_api as R
    from .blip_itm import BlipITM
    if world_size > 1:
        if "OMP_NUM_THREADS" not in os.environ:
            torch.set_num_threads(1)
        ddp_setup(args, rank, world_size)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if not args.bert_vocab:
        raise SystemExit("--real_data needs --bert_vocab (a local bert-base-uncased vocab.txt)")
    tok = data.init_tokenizer(args.bert_vocab)
    cats, nms = data.categories(args, args.coco_annotation_file)
    coco = args.data_type.startswith("coco")
    coco_thing = None
    if args.data_type == "coco_object":      # instance masks need pycocotools, like the reference
        from pycocotools.coco import COCO
        coco_thing = COCO(args.coco_annotation_file)
    if model is None:            # BLIP ITM-large; random init unless --checkpoint names the reference's weights
        torch.manual_seed(4321)
        model = BlipITM(img_size=int(args.img_size), tokenizer=tok).eval()
        if args.checkpoint:
            model.load_lavis_checkpoint(args.checkpoint)
    model.tokenizer = tok
    model = model.to(dev).requires_grad_(False)
    model.gemm_precision = getattr(args, "gemm_precision", "3xfp16")
    ids = data.image_ids(args)
    if args.max_images:
        ids = ids[:int(args.max_images)]
    n_class = (91 if args.data_type == "coco_object" else 183) if coco else len(cats) + 1
    hist0 = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    hist_all = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    wrapped = type("Wrapped", (), {"module": model})()        # the drivers hand a DDP-wrapped model around
    for img_ids in data.batches(ids, args.batch_size, rank, world_size):
        loaded = [data.load_model_image(data.image_path(args, i), args.img_size) for i in img_ids]
        imgs_in = torch.stack([t for t, _, _ in loaded])
        norm_imgs = torch.from_numpy(np.stack([n for _, n, _ in loaded]))
        sizes = [s for _, _, s in loaded]
        head = ([coco_thing] if coco else []) + [wrapped, imgs_in, sizes, args, [None] * len(img_ids), img_ids, args.drop_iter,
                                                 norm_imgs, None, cats, nms, None, rank, args.prune_att_head]
        R.save_img_union_attention(*head, max_block_num=args.max_att_block_num)
        h0, hall = R.save_img_union_attention.last
        if h0 is not None:
            hist0 += h0
        if hall is not None:
            hist_all += hall
    if _fp16_range_exceeded(model, dev, world_size):
        if rank == 0:
            print("warning: an activation left fp16's range in a 3xFP16 GEMM operand; repeating the run with --gemm_precision 3xtf32")
        model.fp16_overflow_flag(dev).zero_()
        args.gemm_precision = "3xtf32"
        if world_size > 1:
            torch.distributed.destroy_process_group()
        return main_real(rank, world_size, args, model=model)
    pipeline.allreduce_hist(hist0)
    pipeline.allreduce_hist(hist_all)
    result = None
    if rank == 0:
        scored = hist_all if int(args.drop_iter) > 1 else hist0
        table, _ = metrics_from_hist(scored.cpu().numpy().astype(np.float64))
        print("images %d  pixAcc %.4f  mAcc %.4f  mIoU %.4f  fwIoU %.4f" % (
            len(ids), table["Pixel Accuracy"], table["Mean Accuracy"], table["Mean IoU"], table["Frequency Weighted IoU"]))
        result = scored.cpu().numpy()
    if world_size > 1:
        torch.distributed.destroy_process_group()
    return result


IMAGE_SUFFIXES = (".jpg", ".jpeg", ".png", ".bmp", ".tif", ".tiff", ".webp")


def wild_images(image_dir):
    """{stem: path} of the image files directly under image_dir.  Two files with one stem are refused: their outputs would
    share a name."""
    paths = {}
    for name in sorted(os.listdir(image_dir)):
        stem, ext = os.path.splitext(name)
        if ext.lower() in IMAGE_SUFFIXES and os.path.isfile(os.path.join(image_dir, name)):
            if stem in paths:
                raise SystemExit("--image_dir holds two images with the stem %r (%s, %s)" % (stem, os.path.basename(paths[stem]), name))
            paths[stem] = os.path.join(image_dir, name)
    if not paths:
        raise SystemExit("no image (%s) in --image_dir %s" % (", ".join(IMAGE_SUFFIXES), image_dir))
    return paths


def parse_class_names(text):
    """'cat, dog,grass' -> ['cat', 'dog', 'grass']."""
    return [c.strip() for c in text.split(",") if c.strip()]


def wild_class_lists(args, stems):
    """{stem: class names} from --classes (one list for every image) or --class_file; at least 1 and at most 255 classes per
    image (the label PNG is 8-bit with 0 for the background)."""
    if bool(args.classes) == bool(args.class_file):
        raise SystemExit("--in_the_wild needs exactly one of --classes and --class_file")
    if args.classes:
        names = parse_class_names(args.classes)
        out = {s: list(names) for s in stems}
    else:
        with open(args.class_file, "r") as f:
            table = json.load(f)
        if not isinstance(table, dict):
            raise SystemExit("--class_file must hold a JSON object {image stem: [class names] or 'a,b,c'}")
        missing = [s for s in stems if s not in table]
        if missing:
            raise SystemExit("--class_file has no classes for %s" % ", ".join(missing))
        out = {s: parse_class_names(table[s]) if isinstance(table[s], str) else [str(c).strip() for c in table[s] if str(c).strip()]
               for s in stems}
    for s, names in out.items():
        if not 1 <= len(names) <= 255:
            raise SystemExit("image %s: %d classes (1 to 255 fit the 8-bit label map)" % (s, len(names)))
    return out


def wild_outputs(save_path, stem):
    """(label PNG, confidence .npy) that --in_the_wild writes for one image."""
    d = os.path.join(save_path, "in_the_wild")
    return os.path.join(d, stem + ".png"), os.path.join(d, stem + "_conf.npy")


def label_palette():
    """The PASCAL VOC colour map (index 0 black): 768 palette bytes."""
    pal = []
    for i in range(256):
        r = g = b = 0
        c = i
        for j in range(8):
            r |= (c & 1) << (7 - j)
            g |= ((c >> 1) & 1) << (7 - j)
            b |= ((c >> 2) & 1) << (7 - j)
            c >>= 3
        pal += [r, g, b]
    return pal


def write_label_png(path, ids):
    from PIL import Image
    im = Image.fromarray(np.ascontiguousarray(ids, dtype=np.uint8))
    im.putpalette(label_palette())
    im.save(path)


def main_in_the_wild(rank, world_size, args, model=None):
    """--in_the_wild: segment_images over this rank's shard of --image_dir, files written per image (no collective).  A 3xFP16
    run whose activations left fp16's range is repeated in 3xTF32 and overwrites its files.  Returns the stems this rank wrote."""
    from .blip_itm import BlipITM
    from .segment import image_size, segment_images, size_refusal
    if args.image_dir is None or args.threshold is None or args.prune_att_head is None:
        raise SystemExit("--in_the_wild needs --image_dir, --threshold and --prune_att_head")
    data_type = args.data_type or "voc"
    paths = wild_images(args.image_dir)
    classes = wild_class_lists(args, list(paths))
    stems = []
    for s in paths:
        why = size_refusal(*image_size(paths[s]), len(classes[s]), args.postprocess, data_type)
        if why:
            if rank == 0:
                print("refused %s: %s" % (paths[s], why))
        else:
            stems.append(s)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if model is None:
        tok = data.init_tokenizer(args.bert_vocab) if args.bert_vocab else synthetic.SyntheticWordPieceTokenizer()
        torch.manual_seed(4321)
        model = BlipITM(img_size=int(args.img_size), tokenizer=tok).eval()
        if args.checkpoint:
            model.load_lavis_checkpoint(args.checkpoint)
        model = model.to(dev).requires_grad_(False)
    model.gemm_precision = getattr(args, "gemm_precision", "3xfp16")
    os.makedirs(os.path.join(args.save_path, "in_the_wild"), exist_ok=True)
    if rank == 0:
        with open(os.path.join(args.save_path, "in_the_wild", "classes.json"), "w") as f:
            json.dump({s: classes[s] for s in stems}, f, indent=1)
    start, end = host.shard_range(len(stems), rank, world_size)
    mine = stems[start:end]
    for b0 in range(0, len(mine), args.batch_size):
        batch = mine[b0:b0 + args.batch_size]
        tic = time.perf_counter()
        res = segment_images(model, [paths[s] for s in batch], [classes[s] for s in batch], img_size=args.img_size, drop_iter=args.drop_iter,
                             threshold=args.threshold, postprocess=args.postprocess, max_att_block_num=args.max_att_block_num,
                             prune_att_head=args.prune_att_head, data_type=data_type, batch_size=len(batch))
        for s, r in zip(batch, res):
            png, conf = wild_outputs(args.save_path, s)
            write_label_png(png, r["ids"])
            if r["conf"] is not None:
                np.save(conf, r["conf"])
        if rank == 0:
            dt = time.perf_counter() - tic
            print("Time: batch of %d images %.4f seconds (%.2f images/s on this rank)" % (len(batch), dt, len(batch) / dt))
    if _fp16_range_exceeded(model, dev, 1):
        print("warning: rank %d: an activation left fp16's range in a 3xFP16 GEMM operand; repeating its images with "
              "--gemm_precision 3xtf32" % rank)
        model.fp16_overflow_flag(dev).zero_()
        args.gemm_precision = "3xtf32"
        return main_in_the_wild(rank, world_size, args, model=model)
    return mine


def main(rank, world_size, args):
    from .blip_itm import BlipITM
    if getattr(args, "in_the_wild", False):
        return main_in_the_wild(rank, world_size, args)
    if getattr(args, "real_data", False):
        return main_real(rank, world_size, args)
    tic = time.perf_counter()
    if world_size > 1:
        # One process per GPU shares the host's cores: with torch's default of one OpenMP worker per core in EVERY rank the
        # spinning workers of one rank starve the kernel-launching thread of the others (measured on 2 GPUs at 150 classes:
        # 2.33 s per batch against 1.58 s with one thread per rank; profiles/diag_two_process_slowdown.sh).  torchrun sets
        # OMP_NUM_THREADS=1 for the same reason; mp.spawn (DRV:1439) does not.
        if "OMP_NUM_THREADS" not in os.environ:
            torch.set_num_threads(1)
        ddp_setup(args, rank, world_size)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    names, n_class = DATASETS[args.data_type]
    tok = synthetic.SyntheticWordPieceTokenizer()
    torch.manual_seed(4321)
    model = BlipITM(img_size=int(args.img_size), tokenizer=tok).to(dev).eval().requires_grad_(False)
    model.gemm_precision = getattr(args, "gemm_precision", "3xfp16")
    layer, head = int(args.max_att_block_num) - 1, int(args.prune_att_head)
    start, end = host.shard_range(args.synthetic_images, rank, world_size)
    items = synthetic_shard(args, names, n_class, start, end)
    hist0 = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    hist_all = torch.zeros((n_class, n_class), dtype=torch.int64, device=dev)
    coco = args.data_type.startswith("coco")
    for b0 in range(0, len(items), args.batch_size):
        batch = items[b0:b0 + args.batch_size]
        tic_batch = time.perf_counter()
        caps = ["A picture of " + " ".join(it["classes"]) for it in batch]                        # DRV:783
        tokens = tok(caps, padding="max_length", max_length=500).to(dev)                          # DRV:317-319
        imgs = torch.stack([it["img"] for it in batch]).to(dev)

        def gradcam_fn(x):
            return model.gradcam(x, caps, tokens, layer=layer, head=head)[0]

        h0, hall, _ = pipeline.batch_confusion(
            gradcam_fn, imgs, tokens.input_ids.tolist(), tok.decode, [it["classes"] for it in batch],
            [[c + 1 for c in it["class_idx"]] for it in batch], [it["gt"] for it in batch], [it["guide"] for it in batch],
            drop_iter=int(args.drop_iter), patch_num=int(int(args.img_size) / 16), threshold=float(args.threshold),
            data_type=args.data_type, mode=args.postprocess, n_class=n_class, coco=coco)
        if h0 is not None:
            hist0 += h0
        if hall is not None:
            hist_all += hall
        if rank == 0:   # batch_confusion ends with a host read of its error flag, so the batch is complete here
            dt = time.perf_counter() - tic_batch
            print("Time: batch of %d images %.4f seconds (%.2f images/s on this rank)" % (len(batch), dt, len(batch) / dt))
    if _fp16_range_exceeded(model, dev, world_size):
        if rank == 0:
            print("warning: an activation left fp16's range in a 3xFP16 GEMM operand; repeating the run with --gemm_precision 3xtf32")
        args.gemm_precision = "3xtf32"
        if world_size > 1:
            torch.distributed.destroy_process_group()
        return main(rank, world_size, args)
    pipeline.allreduce_hist(hist0)
    pipeline.allreduce_hist(hist_all)
    result = None
    if rank == 0:
        first = "syn_%06d" % 0
        if int(args.drop_iter) > 1:
            pipeline.save_hist_npy(hist_all, args.save_path, "all_drop_hist_with_filtered_caption", first, args.max_att_block_num,
                                   args.prune_att_head)
        pipeline.save_hist_npy(hist0, args.save_path, "hist_withfiltered_caption", first, args.max_att_block_num, args.prune_att_head)
        scored = hist_all if int(args.drop_iter) > 1 else hist0
        table, _ = metrics_from_hist(scored.cpu().numpy().astype(np.float64))
        print("images %d  pixAcc %.4f  mAcc %.4f  mIoU %.4f  fwIoU %.4f" % (
            args.synthetic_images, table["Pixel Accuracy"], table["Mean Accuracy"], table["Mean IoU"], table["Frequency Weighted IoU"]))
        print("Time: total running time %.4f seconds" % (time.perf_counter() - tic))
        result = scored.cpu().numpy()
    if world_size > 1:
        torch.distributed.destroy_process_group()
    return result


if __name__ == "__main__":
    import torch.multiprocessing as mp
    args = argparse.ArgumentParser('PnP-OVSS on B200', parents=[get_args_parser()]).parse_args()
    if "RANK" in os.environ:          # launched by torchrun: one rank per process already
        main(int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"]), args)
    elif args.world_size > 1:         # DRV:1439
        mp.spawn(main, args=(args.world_size, args), nprocs=args.world_size)
    else:
        main(0, 1, args)
