"""Images/s through pnp_ovss_b200.segment_images (no ground truth) on 280 seeded JPEG images with a VOC-like size mix (500x375,
375x500, 500x333 and random others; 1-4 classes each), --img_size 336, drop_iter 4, blur+crf, batch 35, the BLIP ITM-large
shape (random init) in the shipped 3xFP16 GEMM mode.  Reports the host load time (decode, resize, tokenize) and the device time
(upload to maps back on the host) apart, with the card name and power limit read in the same run.  One untimed warm-up pass
over the first batch.

    python profiles/time_in_the_wild.py [--images 280] [--out in_the_wild.json]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests", "golden")):
    sys.path.insert(0, p)
import numpy as np
import torch

import synth
from pnp_ovss_b200 import data, segment_images
from pnp_ovss_b200.blip_itm import BlipITM
from pnp_ovss_b200.synthetic import SyntheticWordPieceTokenizer

ap = argparse.ArgumentParser()
ap.add_argument("--images", type=int, default=280)
ap.add_argument("--out", default=None)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("needs a CUDA device")
dev = torch.device("cuda:0")
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                      text=True).stdout.strip()
rng = np.random.default_rng(0)
n = a.images
common = [(375, 500)] * 18 + [(500, 375)] * 7 + [(333, 500)] * 4                    # per 35 images
shapes = [common[i % 35] if i % 35 < len(common) else (int(rng.integers(280, 500)), int(rng.integers(300, 500))) for i in range(n)]
counts = rng.choice([1, 2, 3, 4], size=n, p=[0.55, 0.30, 0.10, 0.05])
class_lists = [sorted(rng.choice(len(data.VOC_NAMES), size=int(c), replace=False).tolist()) for c in counts]
class_lists = [[data.VOC_NAMES[i] for i in cl] for cl in class_lists]
kw = dict(img_size=336, drop_iter=4, threshold=0.15, postprocess="blur+crf", max_att_block_num=8, prune_att_head=9, batch_size=35)
with tempfile.TemporaryDirectory() as tmp:
    from PIL import Image
    paths = []
    for i, (H, W) in enumerate(shapes):
        paths.append(os.path.join(tmp, "img_%04d.jpg" % i))
        Image.fromarray(synth.guide_image(1000 + i, H, W)).save(paths[-1], quality=90)
    torch.manual_seed(4321)
    model = BlipITM(img_size=336, tokenizer=SyntheticWordPieceTokenizer()).to(dev).eval().requires_grad_(False)
    model.gemm_precision = "3xfp16"
    segment_images(model, paths[:35], class_lists[:35], **kw)          # warm-up: module loads, lattice cache, allocator
    torch.cuda.synchronize()
    timings = {}
    tic = time.perf_counter()
    res = segment_images(model, paths, class_lists, timings=timings, **kw)
    wall = time.perf_counter() - tic
    model.check_fp16_overflow()
line = dict(card=card, images=n, img_size=336, batch_size=35, drop_iter=4, postprocess="blur+crf", gemm="3xfp16",
            distinct_shapes=len(set(shapes)), class_counts=np.bincount(counts)[1:].tolist(),
            wall_s=round(wall, 3), images_per_s=round(n / wall, 2), host_load_s=round(timings["load"], 3),
            device_s=round(timings["device"], 3), device_images_per_s=round(n / timings["device"], 2),
            pixels=int(sum(r["ids"].size for r in res)))
print(json.dumps(line))
if a.out:
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(line, f, indent=1)
