"""Host-side inputs of the path for the real datasets: class-name tables, image-id lists, the model-input transform and the
BLIP tokenizer.  Everything here mirrors what the reference's loaders feed into `save_img_union_attention`
(Load_datasets.py = LD, Dataset.py = DS, the LAVIS `BlipBase.init_tokenizer`); none of it touches the GPU.

The datasets, the BERT vocabulary and the BLIP checkpoint are not available offline, so the tests build miniature
directory trees with the same layouts (tests/test_real_data_path.py)."""
import json
import os

import numpy as np
import torch

CLIP_MEAN = (0.48145466, 0.4578275, 0.40821073)   # DS:440
CLIP_STD = (0.26862954, 0.26130258, 0.27577711)

VOC_NAMES = ["aeroplane", "bicycle", "bird", "boat", "bottle", "bus", "car", "cat", "chair", "cow", "table", "dog", "horse",
             "motorbike", "person", "pottedplant", "sheep", "sofa", "train", "tvmonitor"]                        # LD:8-10
CONTEXT_NAMES = ["aeroplane", "bag", "bed", "bedclothes", "bench", "bicycle", "bird", "boat", "book", "bottle", "building",
                 "bus", "cabinet", "car", "cat", "ceiling", "chair", "cloth", "computer", "cow", "cup", "curtain", "dog", "door",
                 "fence", "floor", "flower", "food", "grass", "ground", "horse", "keyboard", "light", "motorbike", "mountain",
                 "mouse", "person", "plate", "platform", "pottedplant", "road", "rock", "sheep", "shelves", "sidewalk", "sign",
                 "sky", "snow", "sofa", "table", "track", "train", "tree", "truck", "tvmonitor", "wall", "water", "window",
                 "wood"]                                                                                        # LD:31-40
ADE_NAMES = ["wall", "building", "sky", "floor", "tree", "ceiling", "road", "bed", "windowpane", "grass", "cabinet", "sidewalk",
             "person", "ground", "door", "table", "mountain", "plant", "curtain", "chair", "car", "water", "painting", "sofa",
             "shelf", "house", "sea", "mirror", "rug", "field", "armchair", "seat", "fence", "desk", "rock", "wardrobe", "lamp",
             "bathtub", "railing", "cushion", "base", "box", "pillar", "signboard", "chest of drawers", "counter", "sand", "sink",
             "skyscraper", "fireplace", "refrigerator", "grandstand", "path", "stairs", "runway", "case", "billiard table",
             "pillow", "screen", "stairway", "river", "bridge", "bookcase", "blind", "coffee table", "toilet", "flower", "book",
             "hill", "bench", "countertop", "stove", "palm", "kitchen island", "computer", "swivel chair", "boat", "bar",
             "arcade machine", "hovel", "bus", "towel", "light", "truck", "tower", "chandelier", "sunshade", "streetlight",
             "booth", "television receiver", "airplane", "dirt track", "apparel", "pole", "land", "bannister", "escalator",
             "ottoman", "bottle", "buffet", "poster", "stage", "van", "ship", "fountain", "conveyer belt", "canopy", "washer",
             "toy", "swimming pool", "stool", "barrel", "basket", "waterfall", "tent", "bag", "motorbike", "cradle", "oven",
             "ball", "food", "stair", "tank", "marque", "microwave", "pot", "animal", "bicycle", "lake", "dishwasher", "screen",
             "blanket", "sculpture", "hood", "sconce", "vase", "trafficlight", "tray", "trash can", "fan", "pier", "crt screen",
             "plate", "monitor", "bulletinboard", "shower", "radiator", "glass", "clock", "flag"]                # LD:61-88


def categories(args, coco_annotation_file=None):
    """(cats, nms) the way the reference's loaders return them: for voc / psc / ade20k a dict {1-based id: name} and the
    caption names (ADE names with their blanks removed, LD:92); for the COCO variants the `categories` list of the
    annotation JSON ([{'id', 'name', ...}], sparse ids) and its names."""
    dt = args.data_type
    if dt in ("voc", "psc", "ade20k"):
        names = {"voc": VOC_NAMES, "psc": CONTEXT_NAMES, "ade20k": ADE_NAMES}[dt]
        cats = {i + 1: n for i, n in enumerate(names)}
        return cats, ["".join(n.split(" ")) for n in names] if dt == "ade20k" else list(names)
    if dt in ("coco_object", "coco_stuff"):
        if coco_annotation_file is None:
            raise ValueError("%s needs the COCO annotation file for its category table" % dt)
        with open(coco_annotation_file, "r") as f:
            cats = sorted(json.load(f)["categories"], key=lambda c: c["id"])
        return cats, [c["name"] for c in cats]
    raise ValueError("unknown data_type %r" % (dt,))


def image_ids(args):
    """The evaluation image ids in file order: voc / psc from `<image dir>/val.txt` (DS:55-76), ade20k from the
    validation .odgt list of semantic-segmentation-pytorch (LD:94; ids are the numeric suffix without padding, which is how
    Load_GroundTruth re-pads them), coco from the file names under coco/images/val2017."""
    dt, home = args.data_type, args.home_dir
    if dt in ("voc", "psc"):
        root = "%s/VOCdevkit/VOC2012" % home if dt == "voc" else "%s/mmsegmentation/data/VOCdevkit/VOC2010" % home
        with open(os.path.join(root, "val.txt"), "r") as f:
            return [line.split(".")[0].strip() for line in f if line.strip()]
    if dt == "ade20k":
        ids = []
        with open("%s/semantic-segmentation-pytorch-master/data/validation.odgt" % home, "r") as f:
            for line in f:
                if line.strip():
                    stem = os.path.splitext(os.path.basename(json.loads(line)["fpath_img"]))[0]      # ADE_val_00000123
                    ids.append(str(int(stem.split("_")[-1])))
        return ids
    if dt in ("coco_object", "coco_stuff"):
        d = "%s/coco/images/val2017/" % home
        return sorted(str(int(os.path.splitext(n)[0])) for n in os.listdir(d) if n.endswith(".jpg"))
    raise ValueError("unknown data_type %r" % (dt,))


def image_path(args, img_id):
    dt, home = args.data_type, args.home_dir
    if dt in ("voc", "psc"):
        return "%s/VOCdevkit/VOC2012/JPEGImages/%s.jpg" % (home, img_id)
    if dt == "ade20k":
        return "%s/ADEChallengeData2016/images/validation/ADE_val_%s.jpg" % (home, str(img_id).rjust(8, "0"))
    return "%s/coco/images/val2017/%012d.jpg" % (home, int(img_id))


def load_model_image(path, img_size):
    """DS:430-443: (model input float32 [3,S,S], norm_img float32 [S,S,3] in 0..1, original (width, height)).
    `path` is an image file, or an RGB image already decoded into a uint8 [H,W,3] array.

    The model input is the image resized to SxS with PIL's bicubic filter, scaled to 0..1 and normalised with the CLIP
    statistics (torchvision Resize(BICUBIC) -> ToTensor -> Normalize on a PIL image is exactly that); norm_img is the
    default-filter resize the reference keeps for its visualisations and the DropOut bookkeeping."""
    from PIL import Image
    img0 = Image.fromarray(path, "RGB") if isinstance(path, np.ndarray) else Image.open(path).convert("RGB")
    S = int(img_size)
    norm_img = np.float32(img0.resize((S, S))) / 255
    x = np.array(img0.resize((S, S), Image.BICUBIC), dtype=np.uint8)
    t = torch.from_numpy(x).permute(2, 0, 1).to(torch.float32).div(255)
    mean = torch.tensor(CLIP_MEAN, dtype=torch.float32).view(3, 1, 1)
    std = torch.tensor(CLIP_STD, dtype=torch.float32).view(3, 1, 1)
    return t.sub_(mean).div_(std), norm_img, img0.size


def init_tokenizer(vocab):
    """The BLIP tokenizer (LAVIS BlipBase.init_tokenizer): bert-base-uncased WordPiece plus the two tokens BLIP appends,
    [DEC] as bos (id 30522) and [ENC] (id 30523, `enc_token_id`, written over [CLS] for the ITM head, BITM:238-239).
    `vocab` is the path of a local vocab.txt (the hub is unreachable offline) or a {token: id} dict."""
    import inspect
    from transformers import BertTokenizer
    if "vocab" in inspect.signature(BertTokenizer.__init__).parameters:      # transformers >= 5
        if isinstance(vocab, str):
            with open(vocab, "r", encoding="utf-8") as f:
                vocab = {line.rstrip("\n"): i for i, line in enumerate(f) if line.rstrip("\n")}
        tok = BertTokenizer(vocab=vocab, do_lower_case=True)
    else:                                                                    # transformers 4.x (the reference pins 4.25)
        tok = BertTokenizer(vocab_file=vocab, do_lower_case=True)
    tok.add_special_tokens({"bos_token": "[DEC]"})
    try:
        tok.add_special_tokens({"additional_special_tokens": ["[ENC]"]})
    except (KeyError, ValueError, AssertionError):
        tok.add_tokens(["[ENC]"], special_tokens=True)
    tok.enc_token_id = tok.convert_tokens_to_ids("[ENC]")
    return tok


def batches(ids, batch_size, rank=0, world_size=1):
    """Contiguous shard of `ids` for this rank (host.shard_range), cut into batches."""
    from .host import shard_range
    start, end = shard_range(len(ids), rank, world_size)
    mine = ids[start:end]
    return [mine[i:i + batch_size] for i in range(0, len(mine), batch_size)]
