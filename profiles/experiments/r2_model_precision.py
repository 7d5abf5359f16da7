"""GradCAM distance from an fp64 autograd pass (4 images, full-size model, block 8 / head 9) and time per 35-image pass for:
native fp32 as torch runs it by default (cuDNN may use TF32 for the patch-embedding convolution), strict fp32 (all TF32 off),
3xTF32 with the corrections in a second GEMM.  (The one-depth-3K-GEMM arm and its switch are at commit 5c46d18.)"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
import bench
from pnp_ovss_b200.blip_itm import BlipITM

dev = torch.device("cuda:0")
w = bench.make_workload(0)
torch.manual_seed(4321)
model = BlipITM(img_size=w["S"], tokenizer=w["tok"]).to(dev).eval().requires_grad_(False)
imgs, caps = w["imgs"].to(dev), w["captions"]
tok = w["tokens"].to(dev)
n = 4
tok4 = w["tok"](caps[:n], padding="max_length", max_length=500).to(dev)
truth = bench.gradcam_fp64(model, imgs[:n].contiguous(), caps[:n], tok4, 7, 9, w["P"])


def run(label):
    for _ in range(2):
        model.gradcam(imgs, caps, tok, layer=7, head=9)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(5):
        model.gradcam(imgs, caps, tok, layer=7, head=9)
    b.record()
    torch.cuda.synchronize()
    got, _ = model.gradcam(imgs[:n].contiguous(), caps[:n], tok4, layer=7, head=9)
    d = (got.double() - truth)
    print("%-44s %.1f ms/pass   GradCAM vs fp64: max %.3e  rms %.3e (of the map's max)" % (
        label, a.elapsed_time(b) / 5, (d.abs().max() / truth.abs().max()).item(), (d.pow(2).mean().sqrt() / truth.abs().max()).item()), flush=True)


model.gemm_precision = "fp32"
run("native fp32 (torch defaults)")
torch.backends.cudnn.allow_tf32 = False
run("strict fp32 (cudnn.allow_tf32 = False)")
torch.backends.cudnn.allow_tf32 = True
model.gemm_precision = "3xtf32"
run("3xtf32, corrections in a second GEMM")
