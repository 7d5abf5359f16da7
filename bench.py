#!/usr/bin/env python
"""bench.py -- images/sec of end-to-end mask extraction (BASELINE.json metric) on N B200s of one node.

A step = one batch of a BASELINE.json configuration (`--config k`, default 1 = "VOC-shaped batch 35 @336, 21 classes,
drop_iter 4, prune_att_head 9, blur+crf", the one the metric is quoted on) through the whole path: the Salience-DropOut
rounds (random-init BLIP ITM-large pass, fused softmax/GradCAM kernel, DropOut kernel), token merge, and -- for every map
the reference driver scores (round-0 and accumulated, DRV:348-403 / 424-481; the COCO driver only the accumulated one,
DRVC:420) -- threshold/upsample, Gaussian blur, dense CRF (10 mean-field iterations), argmax + relabel + confusion matrix.
Data-parallel over images: every rank runs its own batch (weak scaling; `--scaling strong` splits a fixed 280-image list
instead) and the int64 confusion matrices are all-reduced once over NCCL at the end of the timed region.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config k]      # our arm (CUDA kernels through the C ABI)
    python bench.py --impl reference [--steps K] [--warmup W] [--config k] # the reference's CPU path on the host cores

Model GEMMs: by default fp32-grade products on the fp16 tensor cores (`--gemm 3xfp16`, or `3xtf32`: exact hi/lo split of both operands,
three products, fp32 accumulate -- measured closer to an fp64 pass than torch's default fp32 path, see `gemm_accuracy`
in the line); `--gemm fp32` runs torch's native fp32 SIMT GEMMs and is timed beside it as `native_fp32`.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "images/sec end-to-end mask extraction @336"
VOC = ["aeroplane", "bicycle", "bird", "boat", "bottle", "bus", "car", "cat", "chair", "cow", "table", "dog", "horse",
       "motorbike", "person", "plant", "sheep", "sofa", "train", "television"]
COCO_THING_IDS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 27, 28, 31, 32, 33, 34, 35,
                  36, 37, 38, 39, 40, 41, 42, 43, 44, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55, 56, 57, 58, 59, 60, 61, 62, 63, 64, 65,
                  67, 70, 72, 73, 74, 75, 76, 77, 78, 79, 80, 81, 82, 84, 85, 86, 87, 88, 89, 90]
_COMMON = dict(layer=7, head=9, threshold=0.15)
# BASELINE.json configs[k] (SURVEY 8d's concrete inputs).  G = side of ground truth / guide image the maps are upsampled to.
CONFIGS = [
    dict(_COMMON, id=0, name="voc20_b1_336_drop1_blur", B=1, S=336, P=21, G=336, C=20, n_class=21, drop_iter=1, mode="blur",
         data_type="voc", coco=False, baseline="single synthetic 336x336 image, VOC 20 classes, drop_iter 1, blur only"),
    dict(_COMMON, id=1, name="voc21_b35_336_drop4_head9_blur+crf", B=35, S=336, P=21, G=336, C=20, n_class=21, drop_iter=4,
         mode="blur+crf", data_type="voc", coco=False, baseline="VOC-shaped batch 35 @336, 21 classes, drop_iter 4, head 9, blur+crf"),
    dict(_COMMON, id=2, name="ade150_b35_336_drop4_blur+crf", B=35, S=336, P=21, G=336, C=150, n_class=151, drop_iter=4,
         mode="blur+crf", data_type="ade20k", coco=False, baseline="ADE20K-shaped 150 classes @336, batch 35, blur+crf"),
    dict(_COMMON, id=3, name="cocostuff171_b35_336_crf512", B=35, S=336, P=21, G=512, C=171, n_class=183, drop_iter=4,
         mode="blur+crf", data_type="coco_stuff", coco=True,
         baseline="COCO-Stuff-shaped 171 classes @336, dense CRF 10 iterations at full 512x512 resolution"),
    dict(_COMMON, id=4, name="cocoobj81_b35_448_drop4_blur+crf", B=35, S=448, P=28, G=448, C=80, n_class=91, drop_iter=4,
         mode="blur+crf", data_type="coco_object", coco=True, baseline="high-res @448 (28x28 patch grid), COCO-Object 81 classes, drop_iter 4"),
]
WORKLOAD = CONFIGS[1]   # the configuration the metric is quoted on
STRONG_IMAGES = 280     # --scaling strong: a fixed list of 8 batches of 35 split over the ranks


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=range(len(CONFIGS)), help="index into BASELINE.json configs")
    ap.add_argument("--gemm", default="3xfp16", choices=["fp32", "3xtf32", "3xfp16", "tf32", "bf16"],
                    help="the model's torch GEMMs: 3xfp16 (default) / 3xtf32 = fp32-grade error-compensated products on the fp16 / TF32 "
                         "tensor cores (exact hi/lo split of both operands, three products, fp32 accumulate), fp32 = native SIMT fp32; "
                         "tf32 / bf16 are narrower than the reference and only for comparison")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: one batch per rank per step; strong: a fixed %d-image list split over the ranks per step" % STRONG_IMAGES)
    ap.add_argument("--guide", default="natural", choices=["natural", "noise"], help="CRF guide image flavour (SURVEY 8d)")
    ap.add_argument("--ref-images", type=int, default=0, help="images per step of the CPU arm (0 = max(8, cores/2))")
    ap.add_argument("--ref-budget-s", type=float, default=240.0, help="wall-clock budget of the CPU arm's timed steps")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline and ref_gpu legs (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the native-fp32 comparison leg and the fp64 accuracy probe")
    ap.add_argument("--no-parity", action="store_true", help="skip the GPU-vs-oracle label comparison of one bench batch")
    ap.add_argument("--schedule", default="serial", choices=["serial", "overlap", "pipelined"],
                    help="serial (default): everything on one stream; overlap: lattice build + round-0 pass on a second stream under "
                         "DropOut rounds 1..R-1; pipelined: also the accumulated-map pass of batch k under the first model pass of batch "
                         "k+1.  With the model's GEMMs on the tensor cores the part runs at its 1 kW power cap and the serial schedule is "
                         "the fastest (measured A/B/A, --overlap-ab: 371 / 380 / 384 ms per step)")
    ap.add_argument("--overlap-ab", action="store_true", help="also time serial / overlap / pipelined schedules back to back (A/B/A)")
    ap.add_argument("--main-priority", type=int, default=-1,
                    help="CUDA priority of the stream the model passes run on when a second stream is in use (-1: above the "
                         "post-processing stream, so GEMM CTAs are scheduled first; 0: same priority)")
    ap.add_argument("--classes", default="all", choices=["all", "all20", "live"],
                    help="all: every image is captioned with every class of the configuration (BASELINE configs); live (config 1): "
                         "classes per image drawn from the reference's own GPT-4o answers for VOC (mean 1.40)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (float64; rank 0), so "
                         "that two builds run with the same arguments can be compared output for output")
    a = ap.parse_args(argv)
    if a.classes == "all20":
        a.classes = "all"
    a.no_overlap = a.schedule == "serial"
    a.no_pipeline = a.schedule != "pipelined"
    return a


# --------------------------------------------------------------------------------------------------- workload
def class_names(cfg):
    from pnp_ovss_b200 import data
    dt = cfg["data_type"]
    if dt == "voc":
        return list(VOC)
    if dt == "ade20k":
        return ["".join(n.split(" ")) for n in data.ADE_NAMES]
    if dt == "coco_object":
        return ["class%02d" % i for i in range(80)]       # the COCO names live in the (absent) annotation file
    return ["class%03d" % i for i in range(171)]


def class_ids(cfg):
    """Dataset id written for local class i (DRV:392 best_class_idx+1; COCO: the sparse category ids, DRVC:549-584)."""
    dt = cfg["data_type"]
    if dt == "coco_object":
        return list(COCO_THING_IDS)
    if dt == "coco_stuff":
        return list(COCO_THING_IDS) + list(range(92, 183))
    return list(range(1, cfg["C"] + 1))


def make_workload(rank, cfg=None, guide="natural", classes="all", batch_index=0):
    """Seeded synthetic batch of configuration cfg for `rank` (SURVEY 8d); batch_index selects further batches of the same rank."""
    from pnp_ovss_b200 import synthetic as synth
    w = dict(cfg or WORKLOAD)
    B, S, C, n, G = w["B"], w["S"], w["C"], w["n_class"], w["G"]
    seed = rank + 1000 * batch_index
    g = torch.Generator().manual_seed(1234 + seed)
    tok = synth.SyntheticWordPieceTokenizer()
    names, ids_all = class_names(w), class_ids(w)
    if classes == "live":  # the caption the reference really feeds: GPT-4o classes with p > 70 (DRV:764-783)
        if w["data_type"] != "voc":
            raise SystemExit("--classes live is defined for the VOC configurations (the shipped GPT-4o answers)")
        rng = np.random.default_rng(99 + seed)
        counts = rng.choice([1, 2, 3, 4, 6], size=B, p=np.array([983, 366, 88, 11, 1]) / 1449.0)
        idx = [sorted(rng.choice(C, size=int(c), replace=False).tolist()) for c in counts]
        w["name"] = w["name"].replace("voc21", "voc_live_classes")
    else:
        idx = [list(range(C)) for _ in range(B)]
    class_lists = [[names[i] for i in ids] for ids in idx]
    captions = ["A picture of " + " ".join(cl) for cl in class_lists]
    w.update(tok=tok, captions=captions, tokens=tok(captions, padding="max_length", max_length=500),
             class_lists=class_lists, dataset_ids=[[ids_all[i] for i in ids] for ids in idx],
             imgs=torch.randn(B, 3, S, S, generator=g), guide=guide, classes=classes,
             guides=np.stack([synth.guide_image(5000 + 97 * seed + b, G, G, guide) for b in range(B)]),
             gts=np.stack([synth.gt_labels(7000 + 97 * seed + b, G, G, n) for b in range(B)]))
    w["valid_pixels"] = int(((w["gts"] >= 0) & (w["gts"] < n)).sum())
    return w


# --------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.thread = [], None, None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------- roofline bookkeeping
LATTICE_LAUNCHES = {2: 22, 5: 25}  # kernels inside one pnp_lattice_build (see lattice.cu build_impl)
MODEL_KERNELS = {"tf32_split3", "gelu_tf32_split3", "layernorm_tf32_split3", "attention_fp16x3", "softmax_fwd", "softmax_bwd_gradcam"}
# reported in ms, not GB/s: latency-bound classes, the tensor-core-bound attention, and the plain split (launch sizes from 0.1 to 250 MB)
LATENCY_BOUND = {"threshold_prep", "blur_normalize", "lattice_build", "attention_fp16x3", "tf32_split3"}


def channels_of(w):
    from pnp_ovss_b200 import host
    return w["C"] + (1 if host.add_background_rule(w["data_type"], w["C"]) else 0)


def algorithmic_bytes(kernel, w, stats, T, gemm="3xfp16"):
    """Algorithmic bytes per LAUNCH of each custom kernel class (DESIGN.md 'Kernels and rooflines'; SURVEY 8d).  None: the class
    is latency- or tensor-core-bound, or mixes launch sizes (reported in ms only)."""
    op = 6 if gemm == "3xfp16" else 12    # bytes per element of a [hi | lo | hi] GEMM operand
    B, C, P, G = w["B"], w["C"], w["P"], w["G"]
    Cc = channels_of(w)
    N, K = G * G, P * P + 1
    Ms, Mb = stats.get("M_s", 0), stats.get("M_b", 0)
    L = P * P + 1                      # ViT tokens per image
    # blurred modes run the fused low-rank (d) group: the direct separable blur then sees ONE map per image (the background
    # indicator), and only when the configuration has a background channel
    from pnp_ovss_b200 import pipeline as _pl
    lowrank = _pl.USE_LOWRANK_BLUR and P <= 32 and "blur" in (w.get("mode") or "")
    blur_maps = (1 if Cc > C else 0) if lowrank else Cc
    fused_pairs = (Cc + 3) // 4 * 4 <= 112   # crf.cu: two lattice-blur axes per launch up to 448-byte rows
    return {
        "softmax_fwd": 8 * B * 12 * T * K,
        "softmax_bwd_gradcam": 8 * B * (T - 1) * K + 4 * B * (T - 1) * (K - 1),
        "token_merge": 4 * B * (T - 1) * P * P + 4 * B * C * P * P,
        "salience_dropout_round": 4 * B * (T - 1) * P * P * 3 + B * 10 * 3 * 256 * 4,
        "upsample_write": 4 * B * C * P * P + 4 * B * Cc * N,
        "blur_vertical": 8 * B * blur_maps * N or None,
        "blur_horizontal": 8 * B * blur_maps * N or None,
        "crf_unary": 8 * B * Cc * N,
        # SURVEY 8(d) prices the whole (d) group at ONE write of the blurred maps: the fused low-rank kernel reads the PxP grids
        # and writes the unary (pixel-major; the padding channels count in neither figure)
        "lowrank_blur": 4 * B * C * P * P + 4 * B * Cc * N,
        "lowrank_unary": 4 * B * C * P * P + 4 * B * Cc * N,
        "background_blur": 8 * B * N,
        "crf_splat_bilateral": 4 * Cc * (B * N + Mb) + 8 * 6 * B * N,
        # SURVEY 8(d): "2 per blur pass" = one read + one write of the lattice values per axis pass, (d+1) passes.  A fused launch
        # covers two axis passes; the figure is per launch and bench.py also reports the kernel against its REAL traffic.
        "crf_blur_axis_bilateral": (2 if fused_pairs else 1) * (8 * Cc + 8) * Mb,
        "crf_splat_spatial": 4 * Cc * B * (N + Ms) + 8 * 3 * N,
        "crf_blur_axis_spatial": (1.5 if fused_pairs else 1.0) * (8 * Cc + 8) * Ms * B,  # fused: 3 axes in 2 launches (a pair + a single)
        "crf_meanfield_update": 4 * Cc * B * (2 * N) + 4 * Cc * (B * Ms + Mb) + 8 * 9 * B * N,
        "confusion": 12 * B * N,
        "argmax_channels": 4 * Cc * B * N + 4 * B * N,
        # model-pass operand kernels: 4 B read + 12 B written per element ([hi|lo|hi]); sizes vary per call site, the figure is
        # the ViT-L block / MLP shape that dominates each class
        "gelu_tf32_split3": (4 + op) * B * L * 4096,
        "layernorm_tf32_split3": (4 + 4 + 4 + op) * B * L * 1024,   # x and residual in; x and the split out
    }.get(kernel)


def source_fingerprint():
    """sha16 over the CUDA sources: ties profiles/dram_traffic.json (an ncu capture) to the kernels it was measured on."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "pnp_ovss_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(f.encode())
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(kernel, workload_name=None):
    """(per-launch DRAM bytes of `kernel` from the committed ncu capture made by profiles/refresh_traffic.sh, provenance), or
    (None, why) when the capture was made on other kernel sources than the ones built now or on another workload."""
    try:
        j = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
    except (OSError, ValueError):
        return None, "no profiles/dram_traffic.json"
    if j.get("source_sha16") != source_fingerprint():
        return None, "stale: captured on csrc %s, built from %s (run profiles/refresh_traffic.sh)" % (j.get("source_sha16"), source_fingerprint())
    if workload_name is not None and j.get("workload") not in (None, workload_name):
        return None, "captured on workload %s" % j.get("workload")
    v = (j.get("kernels") or {}).get(kernel)
    if not v:
        return None, "kernel not in the capture"
    return v, "ncu dram__bytes_read.sum + dram__bytes_write.sum per launch (%s)" % j.get("captured", "")


def gradcam_fp64(model, imgs, captions, tokens, layer, head, P):
    """GradCAM of (layer, head) from an fp64 copy of the model with plain torch autograd (MED:228-300, BITM:399-433
    restated in torch; no custom kernel) -- the ground truth the GEMM-precision modes are judged against."""
    import copy
    import math
    m = copy.deepcopy(model).double().requires_grad_(True)
    m.gemm_precision = "fp32"
    xa = m.layer[layer].crossattention.self
    kept = {}

    def forward(hidden, enc, enc_mask=None, kv=None, lin=None):
        q, k, v = xa._split(xa.query(hidden)), xa._split(xa.key(enc)), xa._split(xa.value(enc))
        probs = torch.softmax(torch.matmul(q, k.transpose(-1, -2)) / math.sqrt(q.shape[-1]), -1)
        probs.retain_grad()
        kept["probs"] = probs
        ctx = torch.matmul(probs, v)
        B, h, T, d = ctx.shape
        return ctx.permute(0, 2, 1, 3).reshape(B, T, h * d)

    xa.forward = forward
    with torch.enable_grad():
        out = m(imgs.double(), captions)
        out[:, 1].sum().backward()
    p = kept["probs"]
    T = p.shape[2]
    mask = tokens.attention_mask[:, :T].double()
    cam = p[:, head, :, 1:] * p.grad[:, head, :, 1:].clamp(min=0) * mask[:, :, None]
    return cam[:, 1:].reshape(imgs.shape[0], T - 1, P, P).detach()


DTYPE_NAMES = {
    "3xtf32": "f32 (model GEMMs as error-compensated 3xTF32 tensor-core products, fp32 accumulate; custom kernels fp32)",
    "3xfp16": "f32 (model GEMMs as error-compensated 3xFP16 tensor-core products on an exact 22-bit hi/lo split, fp32 accumulate; "
              "custom kernels fp32)",
    "fp32": "f32", "tf32": "tf32 GEMMs (narrower than the reference), fp32 elsewhere", "bf16": "bf16 ViT autocast (narrower than the reference)"}


# --------------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch.distributed as dist
    from pnp_ovss_b200 import _lib, host, pipeline
    from pnp_ovss_b200.blip_itm import BlipITM

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if "OMP_NUM_THREADS" not in os.environ:
            torch.set_num_threads(1)   # one intra-op host thread per rank (DESIGN 8: OpenMP teams of N ranks starve the launch threads)
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    if args.main_priority != 0 and (not args.no_overlap or args.overlap_ab):   # model passes above the post-processing stream: GEMM CTAs are scheduled first
        torch.cuda.set_stream(torch.cuda.Stream(device=dev, priority=args.main_priority))
    cfg = CONFIGS[args.config]
    strong = args.scaling == "strong"
    B = cfg["B"]
    if strong:   # fixed list of STRONG_IMAGES images: rank r owns the batches of its contiguous shard (host.shard_range)
        lo, hi = host.shard_range(STRONG_IMAGES // B, rank, world)
        workloads = [make_workload(0, cfg, args.guide, args.classes, batch_index=i) for i in range(lo, hi)]
    else:
        workloads = [make_workload(rank, cfg, args.guide, args.classes)]
    w = workloads[0] if workloads else make_workload(0, cfg, args.guide, args.classes)
    n_cls = cfg["n_class"]
    torch.manual_seed(4321)  # same random-init weights on every rank
    model = BlipITM(img_size=cfg["S"], tokenizer=w["tok"]).to(dev).eval().requires_grad_(False)
    model.gemm_precision = args.gemm
    if args.gemm == "tf32":
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
    T = max(len(w["tok"].encode(c)) for c in w["captions"])

    pipelined = not args.no_overlap and not args.no_pipeline
    side = pipeline.side_stream(dev)

    class Slot:
        """One batch: pinned host buffers (e2e), resident device copies (value), token tables.  Guide images and ground truth
        are double-buffered on the device: with cross-batch pipelining the post-processing of step k still reads them while
        step k+1's host->device copies arrive."""

        def __init__(self, wl):
            self.w = wl
            self.imgs_h, self.guides_h, self.gts_h = wl["imgs"].pin_memory(), torch.from_numpy(wl["guides"]).pin_memory(), torch.from_numpy(wl["gts"]).pin_memory()
            self.imgs_src = self.imgs_h.to(dev)
            self.imgs_d = torch.empty_like(self.imgs_src)
            self.guides_d = [self.guides_h.to(dev), self.guides_h.to(dev)]
            self.gts_d = [self.gts_h.to(dev), self.gts_h.to(dev)]
            self.free_ev = [None, None]      # side-stream event after which buffer i may be overwritten
            self.turn = 0
            self.tokens_dev = wl["tokens"].to(dev)
            self.token_ids = wl["tokens"].input_ids.tolist()

    slots = [Slot(wl) for wl in workloads]
    total_hist = torch.zeros((n_cls, n_cls), dtype=torch.int64, device=dev)
    hist_host = [torch.empty((n_cls, n_cls), dtype=torch.int64).pin_memory() for _ in range(2)]
    d2h_events = []
    bad = torch.zeros(1, dtype=torch.int32, device=dev)
    last_step = []      # what batch_confusion returned for each batch of the most recent step (--dump-outputs)
    scored = "all_drop" if cfg["drop_iter"] > 1 else "round0"

    def run_batch(s, e2e, stats=None, labels_out=None, overlap=None, defer=False):
        wl = s.w
        i = 0
        if e2e:  # host buffers in
            i = s.turn % 2
            s.turn += 1
            if s.free_ev[i] is not None:     # the batch that last read buffer i (two steps ago) must have finished with it
                torch.cuda.current_stream().wait_event(s.free_ev[i])
            s.imgs_d.copy_(s.imgs_h, non_blocking=True)
            s.guides_d[i].copy_(s.guides_h, non_blocking=True)
            s.gts_d[i].copy_(s.gts_h, non_blocking=True)
        else:    # inputs already resident; DropOut zeroes pixel blocks in place, so restore the working copy
            s.imgs_d.copy_(s.imgs_src)

        def gradcam_fn(x):
            return model.gradcam(x, wl["captions"], s.tokens_dev, layer=cfg["layer"], head=cfg["head"])[0]

        h0, hagg, chosen = pipeline.batch_confusion(gradcam_fn, s.imgs_d, s.token_ids, wl["tok"].decode, wl["class_lists"], wl["dataset_ids"],
                                                    s.gts_d[i], s.guides_d[i], drop_iter=cfg["drop_iter"], patch_num=cfg["P"],
                                                    threshold=cfg["threshold"], data_type=cfg["data_type"], mode=cfg["mode"], coco=cfg["coco"],
                                                    n_class=n_cls, stats=stats, overlap=(not args.no_overlap) if overlap is None else overlap,
                                                    labels_out=labels_out, bad_count=bad, defer=defer)
        if defer and e2e:
            s.free_ev[i] = side.record_event()
        last_step.append({"hist_round0": h0, "hist_all_drop": hagg, "dropout_chosen": chosen})
        return h0, (hagg if hagg is not None else h0)

    def step(e2e, stats=None, serial=False, mode=None):
        """One step: every batch this rank owns (one in weak scaling).  Pipelined: the step returns once its last model pass is
        enqueued; its matrix is folded into the accumulator (and, end to end, copied to the host) on the side stream, and the
        host waits for the PREVIOUS step's copy, so every step's result is read back inside the timed region.
        serial: everything on the main stream, nothing overlapped (the roofline leg: each kernel owns the GPU while it runs)."""
        h = None
        if mode is not None:      # --overlap-ab: force one of the three schedules
            serial, defer = mode == "serial", mode == "pipelined"
        else:
            defer = pipelined and stats is None and not serial
        del last_step[:]
        for s in slots:
            _, h = run_batch(s, e2e, stats, defer=defer, overlap=False if serial else (True if mode is not None else None))
            if defer:
                with torch.cuda.stream(side):
                    total_hist.add_(h)
            else:
                total_hist.add_(h)
        if e2e and h is not None:   # host result out (the step's confusion matrix)
            if defer:
                with torch.cuda.stream(side):
                    hist_host[len(d2h_events) % 2].copy_(h, non_blocking=True)
                    d2h_events.append(side.record_event())
                if len(d2h_events) > 1:
                    d2h_events[-2].synchronize()
            else:
                hist_host[0].copy_(h, non_blocking=True)
                torch.cuda.current_stream().synchronize()
        return h

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(e2e, n_steps, serial=False, mode=None):
        """(ms, reduced int64 matrix of exactly these n_steps).  The all-reduce -- the path's one exchange step -- runs once,
        on a COPY of the accumulator, inside the timed region."""
        total_hist.zero_()
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(n_steps):
            step(e2e, serial=serial, mode=mode)
        pipeline.join_side_stream(dev)           # deferred post-processing of the last steps
        if e2e and d2h_events:
            d2h_events[-1].synchronize()
            del d2h_events[:]
        reduced = total_hist.clone()
        if world > 1:
            dist.all_reduce(reduced, op=dist.ReduceOp.SUM)
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), reduced

    n_ids = lib.pnp_profile_num_kernels()
    tot = (ctypes.c_float * n_ids)()
    cnt = (ctypes.c_int * n_ids)()
    name_of = {i: lib.pnp_profile_kernel_name(i).decode() for i in range(1, n_ids)}

    # ---- warm-up; the last warm-up step is profiled per kernel class to find the dominant custom kernel
    stats = {}
    n_warm = max(args.warmup, 3)
    for i in range(n_warm):
        step(False)
    # One more, profiled, step runs the model pass eagerly: kernels replayed from the model's CUDA graphs are the same launches,
    # but only eager launches pass through the library's event bracketing (and can be counted for `gpu_launches`).  An
    # un-profiled eager step first, so that the caching allocator has its eager-mode blocks before anything is timed.
    graphs_on = (model.USE_VIT_GRAPH, model.USE_TEXT_GRAPH)
    model.USE_VIT_GRAPH = model.USE_TEXT_GRAPH = False
    step(False)
    stats = {"events": []}
    lib.pnp_profile_start(ctypes.c_uint(0xFFFFFFFE))
    step(False, stats)
    torch.cuda.synchronize()
    lib.pnp_profile_stop(tot, cnt, n_ids)
    model.USE_VIT_GRAPH, model.USE_TEXT_GRAPH = graphs_on
    per_kernel = {name_of[i]: (float(tot[i]), int(cnt[i])) for i in range(1, n_ids) if cnt[i]}
    launches_per_step = sum(c for k, (_, c) in per_kernel.items() if k != "lattice_build")
    launches_per_step += per_kernel.get("lattice_build", (0, 0))[1] * LATTICE_LAUNCHES[5]
    ev = stats.pop("events")
    stages = {}
    for (n0, e0), (n1, e1) in zip(ev, ev[1:]):
        stages[n1] = stages.get(n1, 0.0) + e0.elapsed_time(e1)
    # the roofline kernel: the post-processing (SURVEY 8 rows a5-a10) kernel class with the largest total time
    post = [k for k in per_kernel if k not in ("lattice_build", "background_blur") and k not in MODEL_KERNELS]   # (groups of launches)
    dominant = max(post, key=lambda k: per_kernel[k][0])
    dom_id = next(i for i in name_of if name_of[i] == dominant)

    # ---- timed region (inputs resident), dominant kernel bracketed by events in situ
    sampler = ClockSampler(local_rank)
    sampler.start()
    # In the timed region the post-processing runs on the side stream UNDER the model's GEMMs (that is where the throughput
    # comes from), so a launch timed there shares the GPU with a GEMM: reported as `overlapped_avg_launch_ms`.  The roofline
    # itself is taken in a second timed region of the same steps run serially on the main stream, right after: every launch
    # of the dominant kernel is bracketed by events on its own stream and owns the GPU while it runs.
    lib.pnp_profile_filter_stream(ctypes.c_void_p(side.cuda_stream if pipelined else torch.cuda.current_stream().cuda_stream), 1)
    lib.pnp_profile_start(ctypes.c_uint(1 << dom_id))
    ms_total, reduced = timed(False, args.steps)
    timed_outputs = list(last_step)
    lib.pnp_profile_stop(tot, cnt, n_ids)
    lib.pnp_profile_filter_stream(ctypes.c_void_p(0), 0)
    clocks = sampler.stop()
    dom_ms_overlapped = float(tot[dom_id]) / max(int(cnt[dom_id]), 1) if pipelined else None
    if pipelined:
        roof_steps = max(1, min(args.steps, 3))
        lib.pnp_profile_start(ctypes.c_uint(1 << dom_id))
        roof_ms, _ = timed(False, roof_steps, serial=True)
        lib.pnp_profile_stop(tot, cnt, n_ids)
    else:
        roof_steps, roof_ms = args.steps, ms_total
    dom_ms = float(tot[dom_id]) / max(int(cnt[dom_id]), 1)
    dom_launches = int(cnt[dom_id])
    ms_per_step = ms_total / args.steps
    imgs_per_step = (STRONG_IMAGES // B) * B if strong else world * B
    value = imgs_per_step * args.steps / (ms_total / 1e3)

    # ---- optional A/B/A of the three schedules in this process (power-capped parts: overlap is not automatically a win)
    overlap_ab = None
    if args.overlap_ab:
        overlap_ab = {}
        for rep in range(2):
            for mode in ("serial", "overlap", "pipelined"):
                step(False, mode=mode)
                ms, _ = timed(False, args.steps, mode=mode)
                overlap_ab.setdefault(mode, []).append(round(ms / args.steps, 2))

    # ---- the reduced matrix must hold exactly the valid pixels of every rank's every step (a garbage sum cannot pass)
    valid_local = torch.tensor([sum(s.w["valid_pixels"] for s in slots)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(valid_local, op=dist.ReduceOp.SUM)
    hist_total, hist_expected = int(reduced.sum().item()), int(valid_local.item()) * args.steps
    if hist_total != hist_expected:
        raise SystemExit("bench.py: reduced confusion matrix sums to %d, expected %d valid pixels" % (hist_total, hist_expected))
    if int(bad.item()):
        raise SystemExit("bench.py: a relabelled id fell outside [0, n_class)")
    model.check_fp16_overflow()      # 3xFP16 operands: raised if an activation ever left fp16's range (never read per step)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, timed_outputs, reduced)

    # ---- multi-GPU: rank 0 recomputes every rank's shard itself and compares with the all-reduced matrix, bit for bit
    allreduce_check = None
    if world > 1 and not strong:
        per_step = reduced // args.steps
        if rank == 0:
            mine = torch.zeros_like(per_step)
            for r in range(world):
                s = slots[0] if r == 0 else Slot(make_workload(r, cfg, args.guide, args.classes))
                mine += run_batch(s, False)[1]
            torch.cuda.synchronize()
            allreduce_check = {"ok": bool(torch.equal(mine, per_step)), "recomputed_shards": world,
                               "what": "sum over ranks (NCCL all-reduce) / steps == rank 0's own recomputation of all %d shards" % world}
            if not allreduce_check["ok"]:
                raise SystemExit("bench.py: all-reduced confusion matrix differs from the single-rank recomputation")
        dist.barrier()

    # ---- end to end through host buffers
    e2e = None
    if not args.no_e2e:
        step(True)
        e2e_ms, _ = timed(True, args.steps)
        per_batch_h2d = int(w["imgs"].numel() * 4 + w["guides"].size + w["gts"].size * 4)
        e2e = {"value": imgs_per_step * args.steps / (e2e_ms / 1e3), "unit": "images/s",
               "h2d_bytes_per_step": per_batch_h2d * max(len(slots), 1) * world, "d2h_bytes_per_step": int(hist_host[0].numel() * 8) * world,
               "ms_per_step": e2e_ms / args.steps}

    # ---- the same steps on torch's native fp32 SIMT GEMMs, and both modes against an fp64 autograd pass
    native = accuracy = None
    if args.gemm in ("3xtf32", "3xfp16") and not args.no_alt:
        model.gemm_precision = "fp32"
        step(False)
        nat_steps = max(1, min(args.steps, 3))
        nat_ms, _ = timed(False, nat_steps)
        native = {"gemm": "torch native fp32 (cutlass SIMT sgemm), everything else identical", "value": imgs_per_step * nat_steps / (nat_ms / 1e3),
                  "unit": "images/s", "ms_per_step": nat_ms / nat_steps, "steps": nat_steps}
        if rank == 0:
            n = min(4, B)
            probe = slots[0].imgs_src[:n].contiguous()
            tokn = w["tok"](w["captions"][:n], padding="max_length", max_length=500).to(dev)
            cam = {}
            for mode in ("fp32", "3xtf32", "3xfp16"):
                model.gemm_precision = mode
                cam[mode] = model.gradcam(probe, w["captions"][:n], tokn, layer=cfg["layer"], head=cfg["head"])[0]
            torch.backends.cudnn.allow_tf32 = False
            model.gemm_precision = "fp32"
            cam["fp32_strict"] = model.gradcam(probe, w["captions"][:n], tokn, layer=cfg["layer"], head=cfg["head"])[0]
            torch.backends.cudnn.allow_tf32 = True
            try:   # outside any timed region
                truth = gradcam_fp64(model, probe, w["captions"][:n], tokn, cfg["layer"], cfg["head"], cfg["P"])
                sc = truth.abs().max()
                accuracy = {"what": "max |GradCAM - fp64 autograd pass| / max |GradCAM|, %d images, block %d head %d" % (n, cfg["layer"] + 1, cfg["head"]),
                            "3xfp16": float(((cam["3xfp16"].double() - truth).abs().max() / sc).item()),
                            "3xtf32": float(((cam["3xtf32"].double() - truth).abs().max() / sc).item()),
                            "native_fp32_torch_defaults": float(((cam["fp32"].double() - truth).abs().max() / sc).item()),
                            "native_fp32_strict_no_cudnn_tf32": float(((cam["fp32_strict"].double() - truth).abs().max() / sc).item()),
                            "note": "torch's defaults let cuDNN run the patch-embedding convolution in TF32, which is what the reference's "
                                    "GPU path does too; `strict` turns that off"}
                del truth
            except RuntimeError as e:  # e.g. out of memory next to the resident workload: the timings stand
                accuracy = {"error": str(e).splitlines()[0][:120]}
            torch.cuda.empty_cache()
        model.gemm_precision = args.gemm

    # ---- one bench batch's label maps against the oracle fed the SAME saliency maps (rank 0, single GPU)
    parity = None
    if rank == 0 and world == 1 and not args.no_parity and args.classes == "all":
        parity = parity_leg(cfg, slots[0], run_batch)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    uniform = args.classes == "all"
    abytes = algorithmic_bytes(dominant, w, stats, T, args.gemm) if uniform else None  # ragged buckets: no single figure
    achieved = abytes / (dom_ms * 1e-3) / 1e9 if abytes else None
    traffic, traffic_src = measured_traffic(dominant, w["name"])
    roofline = {"kernel": dominant, "bound": "hbm", "achieved": achieved, "peak": peak,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                "frac_on_real_traffic": (traffic / (dom_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "algorithmic_bytes_per_launch": abytes, "avg_launch_ms": dom_ms, "launches_timed": dom_launches,
                "timed_region": ("%d steps run serially on the main stream (%.1f ms per step) right after the pipelined timed region: "
                                 "each launch owns the GPU" % (roof_steps, roof_ms / roof_steps)) if pipelined else
                                "the timed region itself (launches on the main stream)",
                "overlapped_avg_launch_ms": dom_ms_overlapped,
                "share_of_step": per_kernel[dominant][0] / ms_per_step,
                "scope": "largest post-processing kernel class (SURVEY 8 rows a5-a10); every class is listed under `kernels`"}

    cpu_baseline = ref_gpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu_baseline = run_reference_steps(w, n_images=min(B, args.ref_images or default_ref_images()), steps=1, warmup=0, budget_s=60.0)
        try:
            ref_gpu = run_reference_gpu_leg(w, dev, cpu_baseline["cores"])
        except RuntimeError as e:
            ref_gpu = {"unavailable": str(e).splitlines()[0][:160]}

    def kernel_entry(k, v):
        ab = algorithmic_bytes(k, w, stats, T, args.gemm) if uniform else None
        gbps = ab * v[1] / (v[0] * 1e-3) / 1e9 if ab and v[0] > 0 else None
        tr, _ = measured_traffic(k, w["name"])
        return {"ms_per_step": round(v[0], 3), "launches": v[1], "GBps": round(gbps, 1) if gbps else None,
                "frac": round(gbps / peak, 3) if gbps else None,
                "frac_on_real_traffic": round(tr * v[1] / (v[0] * 1e-3) / 1e9 / peak, 3) if tr and v[0] > 0 else None}

    kernels_ms = {k: kernel_entry(k, v) for k, v in sorted(per_kernel.items(), key=lambda kv: -kv[1][0])}
    custom_ms = sum(v[0] for v in per_kernel.values())
    post_ms = sum(v[0] for k, v in per_kernel.items() if k not in MODEL_KERNELS)
    line = {"metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": DTYPE_NAMES[args.gemm], "data": "synthetic",
            "config": {"workload": w["name"], "baseline_config": "configs[%d]: %s" % (cfg["id"], cfg["baseline"]),
                       "images_per_step_per_gpu": B * len(slots), "images_per_step": imgs_per_step, "img_size": cfg["S"], "patch_grid": cfg["P"],
                       "gt_size": cfg["G"], "classes": cfg["C"] if uniform else "live (mean %.2f per image)" % (sum(len(c) for c in w["class_lists"]) / B),
                       "channels": channels_of(cfg) if uniform else "classes + background",
                       "n_class": n_cls, "drop_iter": cfg["drop_iter"], "block": cfg["layer"] + 1,
                       "head": cfg["head"], "postprocess": cfg["mode"], "crf_iters": 10 if "crf" in cfg["mode"] else 0, "tokens_T": T, "guide": args.guide,
                       "model": "BLIP ITM-large shape, random init, torch %s GEMMs, trimmed backward, encoder and text passes replayed "
                                "from CUDA graphs" % args.gemm,
                       "passes": ("all_drop only (DRVC:420)" if cfg["coco"] and cfg["drop_iter"] >= 3 else
                                  "round0 only (drop_iter 1)" if cfg["drop_iter"] == 1 else "round0 + all_drop (DRV:348-403, 424-481)"),
                       "schedule": args.schedule,
                       "overlap": ("off (one stream: fastest on this power-capped part, see --overlap-ab)" if args.no_overlap else
                                   "lattice build + round-0 pass on a side stream under DropOut rounds 1-3" +
                                   ("; accumulated-map pass of step k under the first model pass of step k+1 (main stream priority %d)" % args.main_priority
                                    if pipelined else "")),
                       "parallelism": "dp%d over images" % world, "host_threads_per_rank": torch.get_num_threads(),
                       "M_s": stats.get("M_s"), "M_b_per_batch": stats.get("M_b"),
                       "l2": "per-step working set (>3 GB) exceeds the 126 MB L2; no explicit flush"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches_per_step * args.steps),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "ref_gpu": ref_gpu, "native_fp32": native, "gemm_accuracy": accuracy,
            "parity": parity, "allreduce_check": allreduce_check, "overlap_ab_ms_per_step": overlap_ab,
            "custom_kernels": {"ms_per_step": round(custom_ms, 3), "postprocess_ms_per_step": round(post_ms, 3),
                               "postprocess_images_per_s": round(B * len(slots) / (post_ms * 1e-3), 1) if post_ms else None,
                               "note": "sum of the in-situ event times of every pnp:: kernel in one (warm-up) step, serialised on one "
                                       "stream; the rest of the step is torch's GEMMs / attention"},
            "stages_ms_per_step": {k: round(v, 3) for k, v in stages.items()}, "kernels": kernels_ms,
            "hist_total": hist_total, "hist_expected": hist_expected, "scored_matrix": scored}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, batches, reduced):
    """--dump-outputs: each array batch_confusion returned in the last timed step, the batches of the step stacked on a leading
    axis (hist_round0 / hist_all_drop [batches, n_class, n_class], dropout_chosen [batches, B, 10 * drop_iter]; an array the
    configuration does not produce is not written), and hist_timed_total, the confusion matrix summed over every timed step and
    rank.  float64 holds the int64 counts and the patch indices exactly; the largest case (configs[3], strong scaling) writes
    under 3 MB."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"hist_timed_total": reduced}
    for name, first in batches[0].items():
        if first is not None:
            arrays[name] = torch.stack([b[name] for b in batches])
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


def parity_leg(cfg, slot, run_batch, n_images=4):
    """GPU label maps of one bench batch against the oracle's CPU post-processing (oracle/hotpath.py + the C restatement of
    pydensecrf) fed the SAME class maps: the pixel disagreement rate of this workload.  Outside every timed region."""
    from oracle import reference_arm as RA
    from pnp_ovss_b200 import pipeline
    wl = slot.w
    n = min(n_images, cfg["B"])
    captured = []
    orig = pipeline.merge_tokens_batch

    def spy(gradcam, *a, **k):   # the merged class maps of each pass are what both sides post-process
        out = orig(gradcam, *a, **k)
        captured.append([m.detach().cpu() for m in out[:n]])
        return out

    pipeline.merge_tokens_batch = spy
    labels = {}
    try:
        run_batch(slot, False, labels_out=labels, overlap=False)
        torch.cuda.synchronize()
    finally:
        pipeline.merge_tokens_batch = orig
    names = [k for k in ("round0", "all_drop") if k in labels]
    jobs, keys = [], []
    for name, maps in zip(names, captured):
        rescale = True if name == "round0" else cfg["coco"]
        for b in range(n):
            jobs.append((maps[b].numpy().copy(), cfg["threshold"], (cfg["G"], cfg["G"]), wl["guides"][b], cfg["data_type"],
                         wl["dataset_ids"][b], cfg["mode"], rescale))
            keys.append((name, b))
    pool = RA.make_pool(min(os.cpu_count() or 1, len(jobs)))
    try:
        preds = pool.map(RA._post_one, jobs)
    finally:
        pool.close()
        pool.join()
    out = {"images": n, "what": "GPU relabelled maps vs oracle (CPU) post-processing of the same class maps: fraction of pixels that differ"}
    for name in names:
        diff = tot = 0
        for (nm, b), p in zip(keys, preds):
            if nm == name:
                g = labels[name][b].cpu().numpy()
                diff += int((g != np.asarray(p, dtype=np.float32)).sum())
                tot += g.size
        out[name + "_label_disagreement"] = diff / max(tot, 1)
    return out


# --------------------------------------------------------------------------------------------------- CPU arm
def default_ref_images():
    """Images per CPU step: enough that the per-image post-processing (up to 2 passes each) fills the cores."""
    return max(8, (os.cpu_count() or 1) // 2)


def n_reference_passes(w):
    return 1 if (w["drop_iter"] == 1 or (w["coco"] and w["drop_iter"] >= 3)) else 2


def run_reference_steps(w, n_images, steps, warmup, budget_s=240.0, one_core=False):
    """The reference's CPU path (oracle/reference_arm.py) on the first n_images of the batch; returns the
    cpu_baseline object.  All host threads: torch intra-op threads for the model, one process per (image, pass) afterwards.
    The timed steps stop early (never before one) when `budget_s` of wall clock is spent."""
    from oracle import reference_arm as RA
    from pnp_ovss_b200.blip_itm import BlipITM
    cores = 1 if one_core else (os.cpu_count() or 1)
    torch.set_num_threads(cores)
    torch.manual_seed(4321)
    model = RA.install_reference_capture(BlipITM(img_size=w["S"], tokenizer=w["tok"]).eval())
    n = n_images
    tok = w["tok"]
    tokens = tok(w["captions"][:n], padding="max_length", max_length=500)
    n_passes = n_reference_passes(w)
    workers = 1 if one_core else min(cores, n_passes * n)
    pool = RA.make_pool(workers) if workers > 1 else None
    if pool is not None:
        pool.map(abs, range(workers))  # spin the workers up outside the timed region
    times = []
    timings = {}
    t_begin = time.perf_counter()
    for i in range(warmup + steps):
        if i == warmup:
            timings.clear()
            t_begin = time.perf_counter()
        t0 = time.perf_counter()
        RA.reference_batch_confusion(model, w["imgs"][:n].clone(), w["captions"][:n], tokens, tok.decode, w["class_lists"][:n],
                                     w["dataset_ids"][:n], list(w["gts"][:n]), list(w["guides"][:n]),
                                     drop_iter=w["drop_iter"], layer=w["layer"], head=w["head"], threshold=w["threshold"],
                                     data_type=w["data_type"], mode=w["mode"], n_class=w["n_class"], coco=w["coco"], pool=pool, timings=timings)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
            if time.perf_counter() - t_begin + times[-1] > budget_s:
                break
    if pool is not None:
        pool.close()
        pool.join()
    sec = sum(times) / len(times)
    return {"value": n / sec, "unit": "images/s", "cores": cores, "kind": "port",
            "sample": "%d of the %d images of one batch per step (same seeds), model pass as BITM:386-457 in torch-CPU fp32 "
                      "(12-block capture, full backward), post-processing as DRV:424-481 via oracle/ (scipy gaussian_filter, "
                      "C restatement of pydensecrf), %d reference pass(es) per image fanned over %d worker process(es); %.1f s per step, "
                      "%d timed step(s)" % (n, w["B"], n_passes, workers, sec, len(times)),
            "sec_per_step": sec, "steps_timed": len(times), "images_per_step": n, "model_sec_per_step": timings.get("model_s", 0.0) / len(times),
            "post_sec_per_step": timings.get("post_s", 0.0) / len(times), "post_workers": workers, "post_jobs_per_step": n_passes * n}


def run_reference_gpu_leg(w, dev, cores):
    """The north star's denominator: the model pass on the GPU driven the reference's way (BITM:386-457: capture in all 12
    cross-attention blocks, loss.backward() through ViT-L + BERT with weights requiring grad, 12x12 maps built and copied to
    the host one by one = 144 D2H copies per pass, torch native fp32) followed by the reference's CPU post-processing of the
    whole batch fanned over the host cores (the reference itself uses one core).  One step of the full batch."""
    from oracle import reference_arm as RA
    from pnp_ovss_b200.blip_itm import BlipITM
    torch.manual_seed(4321)
    model = RA.install_reference_capture(BlipITM(img_size=w["S"], tokenizer=w["tok"]).eval()).to(dev)   # parameters require grad
    tok = w["tok"]
    n = w["B"]
    tokens = tok(w["captions"], padding="max_length", max_length=500)
    n_passes = n_reference_passes(w)
    workers = min(cores, n_passes * n)
    pool = RA.make_pool(workers) if workers > 1 else None
    if pool is not None:
        pool.map(abs, range(workers))
    timings = {}
    try:
        for i in range(2):   # one warm-up (cuBLAS/cuDNN plans), one timed
            timings.clear()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            RA.reference_batch_confusion(model, w["imgs"].clone(), w["captions"], tokens, tok.decode, w["class_lists"], w["dataset_ids"],
                                         list(w["gts"]), list(w["guides"]), drop_iter=w["drop_iter"], layer=w["layer"], head=w["head"],
                                         threshold=w["threshold"], data_type=w["data_type"], mode=w["mode"], n_class=w["n_class"],
                                         coco=w["coco"], pool=pool, timings=timings, device=dev)
            sec = time.perf_counter() - t0
        # ... and the way the reference really runs it: ONE process per GPU, post-processing image after image on one core
        # (bounded sample: 4 images)
        n1 = min(4, n)
        tk1 = tok(w["captions"][:n1], padding="max_length", max_length=500)
        t1 = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        torch.set_num_threads(1)
        RA.reference_batch_confusion(model, w["imgs"][:n1].clone(), w["captions"][:n1], tk1, tok.decode, w["class_lists"][:n1], w["dataset_ids"][:n1],
                                     list(w["gts"][:n1]), list(w["guides"][:n1]), drop_iter=w["drop_iter"], layer=w["layer"], head=w["head"],
                                     threshold=w["threshold"], data_type=w["data_type"], mode=w["mode"], n_class=w["n_class"],
                                     coco=w["coco"], pool=None, timings=t1, device=dev)
        sec1 = time.perf_counter() - t0
        torch.set_num_threads(cores)
    finally:
        if pool is not None:
            pool.close()
            pool.join()
        del model
        torch.cuda.empty_cache()
    return {"value": n / sec, "unit": "images/s", "sec_per_step": sec, "images_per_step": n, "model_sec_per_step": timings.get("model_s"),
            "post_sec_per_step": timings.get("post_s"), "post_workers": workers, "cores": cores,
            "single_process": {"value": n1 / sec1, "unit": "images/s", "images": n1, "sec": sec1, "model_sec": t1.get("model_s"),
                               "post_sec": t1.get("post_s"),
                               "what": "the same, as the reference runs it: one process per GPU, post-processing on one core"},
            "what": "reference-style torch-GPU model pass (12-block capture, full backward, 144 D2H per pass, native fp32) + the "
                    "reference's CPU post-processing fanned over %d worker processes (the reference uses 1)" % workers}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    w = make_workload(0, cfg, args.guide, args.classes)
    n = min(cfg["B"], args.ref_images or default_ref_images())
    cb = run_reference_steps(w, n, args.steps, min(args.warmup, 1), budget_s=args.ref_budget_s)
    if not args.no_alt:   # what the reference does per process: one core, one image after the other (bounded: one image, one step)
        oc = run_reference_steps(w, 1, 1, 0, one_core=True)
        cb["one_core"] = {"value": oc["value"], "unit": "images/s", "cores": 1, "sec_per_image": oc["sec_per_step"],
                          "sample": "1 image, 1 step, 1 thread"}
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "images/s",
            "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)), "steps": cb["steps_timed"], "steps_requested": args.steps,
            "warmup": min(args.warmup, 1),
            "ms_per_step": cb["sec_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["name"], "baseline_config": "configs[%d]: %s" % (cfg["id"], cfg["baseline"]), "images_per_step": n,
                       "img_size": w["S"], "gt_size": w["G"], "classes": w["C"], "drop_iter": w["drop_iter"], "postprocess": w["mode"],
                       "device": "host CPU", "note": "a bounded sample of the batch per step; the CPU warm-up is capped at one step and the "
                                                      "timed steps stop at --ref-budget-s"},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
