"""Segmentation of caller-supplied images without ground truth: every image brings its own size and its own class names, and
comes back as a label map (0 = background, i = its i-th class) with, when the post-processing has a CRF, the CRF marginal of
each chosen label.  The images run through the batched GPU path of pipeline.batch_labels; the host only decodes them
(data.load_model_image) and copies the maps back."""
import os
import time

import numpy as np
import torch

from . import data, host, pipeline
from ._lib import PnpError

# pnp_gaussian_blur stages 2 lw halo rows of a column strip in shared memory, lw = int(4 sigma + 0.5) <= 369 at
# sigma = 0.05 max(H, W): the background channel of a blurred mode cannot be blurred on a longer side than this.
BLUR_MAX_SIDE = 1847


def size_refusal(width, height, n_classes, mode, data_type="voc"):
    """The message refusing an image whose maps the blur cannot take (a blurred mode with a background channel and a longer side
    above BLUR_MAX_SIDE), or None when the image can be segmented."""
    if bool(mode) and "blur" in mode and host.add_background_rule(data_type, n_classes) and max(width, height) > BLUR_MAX_SIDE:
        return ("image of %dx%d px: the longer side exceeds the blur's limit of %d px (--postprocess %s with a background channel)"
                % (width, height, BLUR_MAX_SIDE, mode))
    return None


def load_rgb(path_or_array):
    """uint8 [H,W,3] RGB of an image file (any format PIL reads) or of an array ([H,W,3] or [H,W] greyscale, uint8)."""
    if isinstance(path_or_array, np.ndarray):
        a = path_or_array
        if a.dtype != np.uint8 or not (a.ndim == 2 or (a.ndim == 3 and a.shape[2] == 3)):
            raise PnpError("an image array must be uint8 [H,W,3] or [H,W], got %s %s" % (a.dtype, a.shape))
        return np.ascontiguousarray(np.stack([a] * 3, -1) if a.ndim == 2 else a)
    from PIL import Image
    with Image.open(os.fspath(path_or_array)) as im:
        return np.asarray(im.convert("RGB"))


def image_size(path_or_array):
    """(width, height) of an image file (read from its header) or array."""
    if isinstance(path_or_array, np.ndarray):
        return int(path_or_array.shape[1]), int(path_or_array.shape[0])
    from PIL import Image
    with Image.open(os.fspath(path_or_array)) as im:
        return im.size


def caption(classes):
    """'A picture of c1 c2 ...' (DRV:783) with the blanks of a multi-word name removed, so that every class stays one word of
    the caption (as the ADE20K names are, LD:92)."""
    return "A picture of " + " ".join("".join(c.split()) for c in classes)


def segment_images(model, paths_or_arrays, class_lists, *, img_size, drop_iter, threshold, postprocess, max_att_block_num,
                   prune_att_head, data_type="voc", batch_size=35, timings=None):
    """Segment images without ground truth.  model: a BlipITM on the GPU (its .tokenizer tokenizes the captions);
    paths_or_arrays: image files or uint8 RGB arrays; class_lists[i]: the class names of image i.  The model input is
    data.load_model_image's (PIL bicubic resize to img_size, CLIP normalisation); the original RGB image is the CRF guide at its
    own size.  data_type selects the background rule (host.add_background_rule).

    Returns one dict per image: "ids" int32 [H,W] (0 = background, i = class_lists[n][i-1]), "conf" float32 [H,W]
    (the CRF marginal of each chosen label; None when `postprocess` has no CRF) and "classes" (the list given).
    timings (a dict, optional) accumulates "load" (seconds decoding and resizing on the host) and "device" (seconds from the
    upload until the maps are back on the host).

    Raises PnpError before any GPU work for an empty class list or a blank class name, and for an image the blur cannot take (size_refusal)."""
    items = list(paths_or_arrays)
    class_lists = [list(c) for c in class_lists]
    if len(class_lists) != len(items):
        raise PnpError("%d images but %d class lists" % (len(items), len(class_lists)))
    for n, (x, c) in enumerate(zip(items, class_lists)):
        if not c or any(not str(name).split() for name in c):
            raise PnpError("image %d has an empty class list or a blank class name: %r" % (n, c))
        why = size_refusal(*image_size(x), len(c), postprocess, data_type)
        if why:
            raise PnpError("image %d: %s" % (n, why))
    dev = next(model.parameters()).device
    layer, head = int(max_att_block_num) - 1, int(prune_att_head)
    S = int(img_size)
    tok = model.tokenizer
    timings = {} if timings is None else timings
    timings.setdefault("load", 0.0)
    timings.setdefault("device", 0.0)
    out = []
    for b0 in range(0, len(items), int(batch_size)):
        tic = time.perf_counter()
        batch = items[b0:b0 + int(batch_size)]
        classes = class_lists[b0:b0 + int(batch_size)]
        guides = [load_rgb(x) for x in batch]
        loaded = [data.load_model_image(g, S) for g in guides]
        caps = [caption(c) for c in classes]
        tokens = tok(caps, padding="max_length", max_length=500)
        timings["load"] += time.perf_counter() - tic
        tic = time.perf_counter()
        tokens = tokens.to(dev)
        imgs = torch.stack([t for t, _, _ in loaded]).to(dev)

        def gradcam_fn(x):
            return model.gradcam(x, caps, tokens, layer=layer, head=head)[0]

        maps = pipeline.batch_labels(gradcam_fn, imgs, tokens.input_ids.tolist(), tok.decode, classes, guides, drop_iter=int(drop_iter),
                                     patch_num=S // 16, threshold=float(threshold), data_type=data_type, mode=postprocess)
        for (ids, conf), c in zip(maps, classes):
            out.append(dict(ids=ids.cpu().numpy(), conf=conf.cpu().numpy() if conf is not None else None, classes=c))
        timings["device"] += time.perf_counter() - tic
    return out
