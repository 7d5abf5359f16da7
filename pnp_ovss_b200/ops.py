"""Tensor-level wrappers over the C ABI: one Python function per entry point of include/pnp_ovss_b200.h.

PyTorch is used for device memory and streams only: every function takes CUDA tensors, passes raw pointers and
the current stream to libpnp_ovss_b200.so and returns CUDA tensors.  Non-CUDA inputs raise (no CPU fallback)."""
import ctypes

import torch

from . import _lib
from ._lib import PnpError, check


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _req(t, dtype, name, ndim=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise PnpError("%s must be a CUDA tensor (pnp_ovss_b200 has no CPU path)" % name)
    if t.dtype != dtype:
        raise PnpError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise PnpError("%s must be contiguous" % name)
    if ndim is not None and t.dim() != ndim:
        raise PnpError("%s must have %d dims, got %s" % (name, ndim, tuple(t.shape)))
    return t


# ----------------------------------------------------------------------------------------------- (a)
def softmax_fwd(scores, key_mask=None, scale=0.125, out=None):
    """probs = softmax(scores*scale + key_mask, -1); scores [B,h,T,K] (MED:267-274)."""
    _req(scores, torch.float32, "scores", 4)
    B, h, T, K = scores.shape
    if key_mask is not None:
        _req(key_mask, torch.float32, "key_mask", 2)
        if tuple(key_mask.shape) != (B, K):
            raise PnpError("key_mask must be [B,K]")
    probs = torch.empty_like(scores) if out is None else _req(out, torch.float32, "out", 4)
    check(_lib.load().pnp_xattn_softmax_fwd(_p(scores), _p(key_mask), _p(probs), B, h, T, K, float(scale), _stream()),
          "pnp_xattn_softmax_fwd")
    return probs


def softmax_bwd_gradcam(probs, dprobs, token_mask, head, scale=0.125, need_dscores=True, need_gradcam=True):
    """(dscores or None, gradcam [B,T-1,K-1] or None); see pnp_xattn_softmax_bwd_gradcam (BITM:415-433)."""
    _req(probs, torch.float32, "probs", 4)
    _req(dprobs, torch.float32, "dprobs", 4)
    if probs.shape != dprobs.shape:
        raise PnpError("probs/dprobs shape mismatch")
    B, h, T, K = probs.shape
    dscores = torch.empty_like(probs) if need_dscores else None
    gradcam = None
    stride = 0
    if need_gradcam:
        _req(token_mask, torch.int64, "token_mask", 2)
        if token_mask.shape[0] != B or token_mask.shape[1] < T:
            raise PnpError("token_mask must be [B, >=T]")
        stride = token_mask.shape[1]
        gradcam = torch.empty((B, T - 1, K - 1), dtype=torch.float32, device=probs.device)
        if not 0 <= int(head) < h:
            raise PnpError("head out of range")
    if all(t is None or t.numel() == 0 for t in (dscores, gradcam)):
        # nothing to write (B == 0, or frozen mode with T == 1): an empty tensor's null data pointer would read as "output not
        # requested" to the library, which refuses a call that requests no output
        return dscores, gradcam
    check(_lib.load().pnp_xattn_softmax_bwd_gradcam(_p(probs), _p(dprobs), _p(dscores), _p(token_mask if need_gradcam else None),
                                                    stride, _p(gradcam), B, h, T, K, float(scale), int(head), _stream()),
          "pnp_xattn_softmax_bwd_gradcam")
    return dscores, gradcam


# ----------------------------------------------------------------------------------------------- (b)
def token_merge(gradcam, seg_start, seg_len, seg_div, row_offset=3, max_end=None):
    """gradcam [B,Tm,P,P] or [B,Tm,PP]; seg_* [B,C] -> class maps [B,C,*spatial] (DRV:810-853).
    max_end = max(seg_start + seg_len), known to the host code that built the tables (pipeline.segment_tensors); when it
    is not given the bound is read back from the device (a blocking copy: tests and one-off calls only)."""
    _req(gradcam, torch.float32, "gradcam")
    B, Tm = gradcam.shape[:2]
    spatial = tuple(gradcam.shape[2:])
    PP = 1
    for s in spatial:
        PP *= s
    _req(seg_start, torch.int32, "seg_start", 2)
    _req(seg_len, torch.int32, "seg_len", 2)
    _req(seg_div, torch.float32, "seg_div", 2)
    C = seg_start.shape[1]
    if max_end is None:
        max_end = int((seg_start + seg_len).max())
    if int(max_end) + row_offset > Tm:
        raise PnpError("token segment runs past the GradCAM rows")
    out = torch.empty((B, C) + spatial, dtype=torch.float32, device=gradcam.device)
    check(_lib.load().pnp_token_merge(_p(gradcam), _p(seg_start), _p(seg_len), _p(seg_div), _p(out), B, Tm, PP, C, row_offset,
                                      _stream()), "pnp_token_merge")
    return out


# ----------------------------------------------------------------------------------------------- (c)
def salience_dropout_round(gradcam, agg, chosen, n_prev, imgs, norm_imgs, P, patch, row_lo, row_hi, save_len, round_idx,
                           ensemble_r=None):
    """One Salience DropOut round, in place on agg / chosen / imgs / norm_imgs (DRV:589-647, 716-721)."""
    _req(gradcam, torch.float32, "gradcam")
    B, Tm = gradcam.shape[:2]
    _req(chosen, torch.int32, "chosen", 2)
    if chosen.shape[0] != B or chosen.shape[1] < int(n_prev) + int(save_len):
        raise PnpError("chosen must be [B, >= n_prev + save_len]")
    if gradcam.numel() != B * Tm * P * P:
        raise PnpError("gradcam must be [B,Tm,P,P]")
    if agg is not None:
        _req(agg, torch.float32, "agg")
        if agg.shape != gradcam.shape:
            raise PnpError("agg must have gradcam's shape")
    if imgs is not None:
        _req(imgs, torch.float32, "imgs", 4)
        if tuple(imgs.shape) != (B, 3, P * patch, P * patch):
            raise PnpError("imgs must be [B,3,P*patch,P*patch]")
    if norm_imgs is not None:      # the kernel writes norm_imgs[((b*S+y)*S+x)*3+ch]: anything but [B,S,S,3] would be written out of bounds
        _req(norm_imgs, torch.float32, "norm_imgs", 4)
        if tuple(norm_imgs.shape) != (B, P * patch, P * patch, 3):
            raise PnpError("norm_imgs must be [B,P*patch,P*patch,3]")
    if ensemble_r is not None:
        _req(ensemble_r, torch.float32, "ensemble_r")
        if ensemble_r.shape != gradcam.shape:
            raise PnpError("ensemble_r must have gradcam's shape")
    check(_lib.load().pnp_salience_dropout_round(_p(gradcam), _p(ensemble_r), _p(agg), _p(chosen), chosen.shape[1], int(n_prev),
                                                 _p(imgs), _p(norm_imgs), B, Tm, int(P), int(patch), int(row_lo), int(row_hi),
                                                 int(save_len), int(round_idx), _stream()), "pnp_salience_dropout_round")


# ----------------------------------------------------------------------------------------------- (d)
def threshold_upsample(class_maps, H, W, threshold, rescale, with_background):
    """class_maps [B,C,P,P] -> [B,C',H,W] (DRV:424-455 / DRV:348-380)."""
    _req(class_maps, torch.float32, "class_maps", 4)
    B, C, P, _ = class_maps.shape
    lib = _lib.load()
    ws_bytes = lib.pnp_threshold_upsample_workspace_bytes(B, C, P)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=class_maps.device)
    out = torch.empty((B, C + (1 if with_background else 0), H, W), dtype=torch.float32, device=class_maps.device)
    check(lib.pnp_threshold_upsample(_p(class_maps), _p(out), _p(ws), ws_bytes, B, C, P, int(H), int(W), float(threshold),
                                     int(bool(rescale)), int(bool(with_background)), _stream()), "pnp_threshold_upsample")
    return out


def gaussian_blur(maps, sigma, normalize=True):
    """maps [..., H, W] -> (blurred, minmax [n_maps,2]); scipy.ndimage.gaussian_filter semantics (DRV:1149-1153)."""
    _req(maps, torch.float32, "maps")
    H, W = maps.shape[-2:]
    n_maps = maps.numel() // (H * W)
    lib = _lib.load()
    ws_bytes = lib.pnp_gaussian_blur_workspace_bytes(n_maps, H, W, float(sigma))
    if ws_bytes == 0:
        raise PnpError("unsupported blur configuration (sigma=%r, H=%d, W=%d)" % (sigma, H, W))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=maps.device)
    out = torch.empty_like(maps)
    minmax = torch.empty((n_maps, 2), dtype=torch.float32, device=maps.device)
    check(lib.pnp_gaussian_blur(_p(maps), _p(out), _p(minmax), _p(ws), ws_bytes, n_maps, H, W, float(sigma), int(bool(normalize)),
                                _stream()), "pnp_gaussian_blur")
    return out, minmax


def lowrank_blur_unary(class_maps, H, W, threshold, rescale, with_background, sigma, unary=True, labels=False, maps=False, minmax=False,
                       n_classes=None):
    """Fused threshold -> upsample -> background -> blur -> min-max -> {CRF unary | argmax labels | maps} for class_maps
    [B,C,P,P] (pnp_lowrank_blur_unary).  Returns a dict with the requested outputs: "unary" [B,N,Cp], "labels" int32 [B,N],
    "maps" [B,C',H,W], "minmax" [B*C',2].
    n_classes: int32 [B] CUDA tensor for a batch PADDED to C classes (pnp_lowrank_blur_unary_padded): image b has n_classes[b] <= C
    classes; its other channels, and the padding up to Cp, come out dead (unary +inf), ready for crf_inference(C = Cp)."""
    _req(class_maps, torch.float32, "class_maps", 4)
    B, C, P, P2 = class_maps.shape
    if P != P2:
        raise PnpError("class_maps must be [B,C,P,P]")
    if n_classes is not None:
        _req(n_classes, torch.int32, "n_classes", 1)
        if n_classes.shape[0] != B:
            raise PnpError("n_classes must be [B]")
    lib = _lib.load()
    ws_bytes = lib.pnp_lowrank_blur_workspace_bytes(B, C, P, int(H), int(W), float(sigma), int(bool(with_background)))
    if ws_bytes == 0:
        raise PnpError("unsupported low-rank blur configuration (P=%d, H=%d, W=%d, sigma=%r)" % (P, H, W, sigma))
    dev = class_maps.device
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    Cc = C + (1 if with_background else 0)
    N = int(H) * int(W)
    out = {}
    if unary:
        out["unary"] = torch.empty((B, N, crf_pad_channels(Cc)), dtype=torch.float32, device=dev)
    if labels:
        out["labels"] = torch.empty((B, N), dtype=torch.int32, device=dev)
    if maps:
        out["maps"] = torch.empty((B, Cc, int(H), int(W)), dtype=torch.float32, device=dev)
    if minmax:
        out["minmax"] = torch.empty((B * Cc, 2), dtype=torch.float32, device=dev)
    if not (unary or labels or maps):
        raise PnpError("nothing to compute")
    check(lib.pnp_lowrank_blur_unary_padded(_p(class_maps), _p(n_classes), _p(out.get("unary")), _p(out.get("labels")), _p(out.get("maps")),
                                            _p(out.get("minmax")), _p(ws), ws_bytes, B, C, P, int(H), int(W), float(threshold),
                                            int(bool(rescale)), int(bool(with_background)), float(sigma), _stream()),
          "pnp_lowrank_blur_unary_padded")
    return out


# ----------------------------------------------------------------------------------------------- (e)
class LatticeHandle:
    """A finished permutohedral lattice in device memory (owns its storage tensor)."""

    def __init__(self, d, n_images, H, W, shared, device):
        lib = _lib.load()
        self.H, self.W = int(H), int(W)
        self.struct = _lib.Lattice()
        nbytes = lib.pnp_lattice_storage_bytes(d, n_images, H * W)
        if nbytes == 0:
            raise PnpError("bad lattice shape")
        self.storage = torch.empty(nbytes + 256, dtype=torch.uint8, device=device)
        base = (self.storage.data_ptr() + 255) // 256 * 256
        self._base = base
        check(lib.pnp_lattice_init(ctypes.byref(self.struct), ctypes.c_void_p(base), nbytes, d, n_images, H * W, int(shared)),
              "pnp_lattice_init")

    @property
    def M(self):
        return self.struct.n_vertices

    @property
    def d(self):
        return self.struct.d

    def _view(self, field, count, dtype):
        off = getattr(self.struct, field) - self.storage.data_ptr()
        itemsize = torch.empty((), dtype=dtype).element_size()
        return self.storage[off:off + count * itemsize].view(dtype)

    def arrays(self):
        """Device views (for tests): offset [n_lp,d+1], bary, nbr [d+1,M,2], norm [n_lp], row_ptr, csr_pix, csr_w, csr_norm."""
        s = self.struct
        n_lp = s.n_images * s.n_pixels
        D1 = s.d + 1
        ne = n_lp * D1
        return {
            "offset": self._view("offset", ne, torch.int32).view(n_lp, D1),
            "bary": self._view("bary", ne, torch.float32).view(n_lp, D1),
            "nbr": self._view("nbr", D1 * s.vertex_stride * 2, torch.int32).view(D1, s.vertex_stride, 2)[:, :s.n_vertices],
            "norm": self._view("norm", n_lp, torch.float32),
            "row_ptr": self._view("row_ptr", s.n_vertices + 1, torch.int32),
            "csr_pix": self._view("csr_pix", ne, torch.int32),
            "csr_w": self._view("csr_w", ne, torch.float32),
            "csr_norm": self._view("csr_norm", ne, torch.float32),
        }


def build_lattice_begin(H, W, sxy, rgb=None, srgb=None, device=None):
    """Enqueue the build of a spatial lattice (rgb None; shared by every image of a batch) or of a bilateral lattice over rgb uint8
    [B,H,W,3] on the current stream (pnp_lattice_build, asynchronous).  Returns (handle, workspace) for build_lattice_finish."""
    lib = _lib.load()
    sx, sy = (sxy, sxy) if not isinstance(sxy, (tuple, list)) else sxy
    if rgb is None:
        if device is None:
            raise PnpError("device required for a spatial lattice")
        lat = LatticeHandle(2, 1, H, W, True, device)
        sr = sg = sb = 1.0
    else:
        _req(rgb, torch.uint8, "rgb", 4)
        if tuple(rgb.shape[1:]) != (H, W, 3):
            raise PnpError("rgb must be [B,H,W,3] uint8")
        sr, sg, sb = (srgb, srgb, srgb) if not isinstance(srgb, (tuple, list)) else srgb
        lat = LatticeHandle(5, rgb.shape[0], H, W, False, rgb.device)
        device = rgb.device
    s = lat.struct
    ws_bytes = lib.pnp_lattice_build_workspace_bytes(s.d, s.n_images, s.n_pixels)
    ws = torch.empty(ws_bytes + 256, dtype=torch.uint8, device=device)
    ws_base = (ws.data_ptr() + 255) // 256 * 256
    check(lib.pnp_lattice_build(ctypes.byref(s), _p(rgb), int(H), int(W), float(sx), float(sy), float(sr), float(sg), float(sb),
                                ctypes.c_void_p(ws_base), ws_bytes, _stream()), "pnp_lattice_build")
    return lat, ws


def build_lattice_finish(lat, ws):
    """Second half of a build (pnp_lattice_finish: waits for the stream the build was enqueued on -- call it under that stream --
    and reads the vertex count back).  Several builds enqueued on different streams overlap when their finishes come afterwards."""
    check(_lib.load().pnp_lattice_finish(ctypes.byref(lat.struct), _stream()), "pnp_lattice_finish")
    del ws
    return lat


def build_lattice(H, W, sxy, rgb=None, srgb=None, device=None):
    """Spatial lattice (rgb None; shared by every image of a batch) or bilateral lattice over rgb uint8 [B,H,W,3]."""
    return build_lattice_finish(*build_lattice_begin(H, W, sxy, rgb=rgb, srgb=srgb, device=device))


def _lattice_array(lattices):
    arr = (ctypes.POINTER(_lib.Lattice) * len(lattices))(*[ctypes.pointer(l.struct) for l in lattices])
    return arr


def crf_pad_channels(C):
    return (C + 3) // 4 * 4


def crf_unary_from_maps(maps, minmax=None):
    """maps [B,C,N] (blurred, un-normalised if minmax given) -> unary [B,N,Cp] (DRV:1057-1063)."""
    _req(maps, torch.float32, "maps", 3)
    B, C, N = maps.shape
    if minmax is not None:
        _req(minmax, torch.float32, "minmax")
    U = torch.empty((B, N, crf_pad_channels(C)), dtype=torch.float32, device=maps.device)
    lib = _lib.load()
    ws_bytes = lib.pnp_crf_unary_workspace_bytes(B, C, N)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=maps.device) if ws_bytes else None
    check(lib.pnp_crf_unary_from_maps(_p(maps), _p(minmax), _p(U), _p(ws), ws_bytes, B, C, N, _stream()), "pnp_crf_unary_from_maps")
    return U


def crf_pack(x_cn):
    """[B,C,N] -> [B,N,Cp]."""
    _req(x_cn, torch.float32, "x", 3)
    B, C, N = x_cn.shape
    out = torch.empty((B, N, crf_pad_channels(C)), dtype=torch.float32, device=x_cn.device)
    check(_lib.load().pnp_crf_pack_cn_to_nc(_p(x_cn), _p(out), B, C, N, _stream()), "pnp_crf_pack_cn_to_nc")
    return out


def crf_unpack(x_nc, C):
    """[B,N,Cp] -> [B,C,N]."""
    _req(x_nc, torch.float32, "x", 3)
    B, N, Cp = x_nc.shape
    if Cp != crf_pad_channels(C):
        raise PnpError("channel padding mismatch")
    out = torch.empty((B, C, N), dtype=torch.float32, device=x_nc.device)
    check(_lib.load().pnp_crf_unpack_nc_to_cn(_p(x_nc), _p(out), B, C, N, _stream()), "pnp_crf_unpack_nc_to_cn")
    return out


def crf_filter(lattice, x_nc, normalized=True):
    """y = norm.K(norm.x) (or K x) over one lattice; x [B,N,Cp]."""
    _req(x_nc, torch.float32, "x", 3)
    B, N, Cp = x_nc.shape
    lib = _lib.load()
    arr = _lattice_array([lattice])
    nbytes = lib.pnp_crf_scratch_bytes(arr, 1, B, Cp)
    if nbytes == 0:
        raise PnpError("lattice/batch mismatch")
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=x_nc.device)
    y = torch.empty_like(x_nc)
    check(lib.pnp_crf_filter(ctypes.byref(lattice.struct), _p(x_nc), _p(y), _p(scratch), nbytes, B, Cp, int(bool(normalized)),
                             _stream()), "pnp_crf_filter")
    return y


def crf_inference(lattices, weights, unary, C, n_iter, want_labels=True, scratch=None):
    """Mean-field inference; unary [B,N,Cp] -> (Q [B,N,Cp], labels int32 [B,N] or None)."""
    _req(unary, torch.float32, "unary", 3)
    B, N, Cp = unary.shape
    lib = _lib.load()
    arr = _lattice_array(lattices)
    nbytes = lib.pnp_crf_scratch_bytes(arr, len(lattices), B, Cp)
    if nbytes == 0:
        raise PnpError("lattice/batch mismatch")
    if scratch is None or scratch.numel() < nbytes:
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=unary.device)
    Q = torch.empty_like(unary)
    labels = torch.empty((B, N), dtype=torch.int32, device=unary.device) if want_labels else None
    w = (ctypes.c_float * len(weights))(*[float(x) for x in weights])
    check(lib.pnp_crf_inference(arr, w, len(lattices), _p(unary), _p(Q), _p(scratch), scratch.numel(), _p(labels), B, int(C), Cp,
                                int(n_iter), _stream()), "pnp_crf_inference")
    return Q, labels


# ----------------------------------------------------------------------------------------------- (f)1 model-pass GEMM operands
def tf32_split3(x):
    """x [..., K] -> [..., 3K] = [hi | lo | hi] (exact TF32 split; see pnp_tf32_split3)."""
    _req(x, torch.float32, "x")
    K = x.shape[-1]
    M = x.numel() // K
    out = torch.empty(x.shape[:-1] + (3 * K,), dtype=torch.float32, device=x.device)
    check(_lib.load().pnp_tf32_split3(_p(x), _p(out), M, K, _stream()), "pnp_tf32_split3")
    return out


def gelu_tf32_split3(x, bias=None):
    """[hi | lo | hi] split of GELU(x + bias) (exact erf form)."""
    _req(x, torch.float32, "x")
    K = x.shape[-1]
    M = x.numel() // K
    if bias is not None:
        _req(bias, torch.float32, "bias", 1)
        if bias.shape[0] != K:
            raise PnpError("bias must be [K]")
    out = torch.empty(x.shape[:-1] + (3 * K,), dtype=torch.float32, device=x.device)
    check(_lib.load().pnp_gelu_tf32_split3(_p(x), _p(bias), _p(out), M, K, _stream()), "pnp_gelu_tf32_split3")
    return out


def layernorm_tf32_split3(x, gamma, beta, eps, residual=None, residual_bias=None, split=True, plain=False):
    """LayerNorm over the last dim of x (or of x + residual + residual_bias, which then REPLACES x in place).
    Returns (split [..., 3K] or None, plain [..., K] or None)."""
    _req(x, torch.float32, "x")
    K = x.shape[-1]
    M = x.numel() // K
    _req(gamma, torch.float32, "gamma", 1)
    _req(beta, torch.float32, "beta", 1)
    if gamma.shape[0] != K or beta.shape[0] != K:
        raise PnpError("gamma/beta must be [K]")
    if residual is not None:
        _req(residual, torch.float32, "residual")
        if residual.shape != x.shape:
            raise PnpError("residual shape mismatch")
    if residual_bias is not None:
        _req(residual_bias, torch.float32, "residual_bias", 1)
        if residual is None or residual_bias.shape[0] != K:
            raise PnpError("residual_bias needs a residual and must be [K]")
    if not (split or plain):
        raise PnpError("nothing to compute")
    out3 = torch.empty(x.shape[:-1] + (3 * K,), dtype=torch.float32, device=x.device) if split else None
    out1 = torch.empty_like(x) if plain else None
    check(_lib.load().pnp_layernorm_tf32_split3(_p(x), _p(residual), _p(residual_bias), _p(x if residual is not None else None),
                                                _p(gamma), _p(beta), float(eps), _p(out3), _p(out1), M, K, _stream()),
          "pnp_layernorm_tf32_split3")
    return out3, out1


def fp16_split3(x, in_scale=1.0, hi_scale=1.0, flag=None):
    """x [..., K] fp32 -> fp16 [..., 3K] = [h*hi_scale | (x-h)*2^11 | h] of x*in_scale (pnp_fp16_split3)."""
    _req(x, torch.float32, "x")
    K = x.shape[-1]
    M = x.numel() // K
    out = torch.empty(x.shape[:-1] + (3 * K,), dtype=torch.float16, device=x.device)
    check(_lib.load().pnp_fp16_split3(_p(x), float(in_scale), float(hi_scale), _p(out), _p(flag), M, K, _stream()), "pnp_fp16_split3")
    return out


def gelu_fp16_split3(x, bias=None, in_scale=1.0, hi_scale=1.0, flag=None):
    """fp16 [h*hi_scale | l | h] split of GELU(x*in_scale + bias) (exact erf form)."""
    _req(x, torch.float32, "x")
    K = x.shape[-1]
    M = x.numel() // K
    if bias is not None:
        _req(bias, torch.float32, "bias", 1)
        if bias.shape[0] != K:
            raise PnpError("bias must be [K]")
    out = torch.empty(x.shape[:-1] + (3 * K,), dtype=torch.float16, device=x.device)
    check(_lib.load().pnp_gelu_fp16_split3(_p(x), float(in_scale), _p(bias), float(hi_scale), _p(out), _p(flag), M, K, _stream()),
          "pnp_gelu_fp16_split3")
    return out


def layernorm_fp16_split3(x, gamma, beta, eps, residual=None, residual_scale=1.0, residual_bias=None, hi_scale=1.0, split=True,
                          plain=False, flag=None, bias_one=None):
    """LayerNorm over the last dim of x (or of x + residual*residual_scale + residual_bias, which then REPLACES x in place).
    Returns (fp16 split [..., 3K] or None, plain fp32 [..., K] or None).  bias_one: append the 8 bias columns
    [bias_one, 1, 0 x 6] to every row of the split ([..., 3K + 8]) so that the GEMM adds the next layer's bias itself."""
    _req(x, torch.float32, "x")
    K = x.shape[-1]
    M = x.numel() // K
    _req(gamma, torch.float32, "gamma", 1)
    _req(beta, torch.float32, "beta", 1)
    if gamma.shape[0] != K or beta.shape[0] != K:
        raise PnpError("gamma/beta must be [K]")
    if residual is not None:
        _req(residual, torch.float32, "residual")
        if residual.shape != x.shape:
            raise PnpError("residual shape mismatch")
    if residual_bias is not None:
        _req(residual_bias, torch.float32, "residual_bias", 1)
        if residual is None or residual_bias.shape[0] != K:
            raise PnpError("residual_bias needs a residual and must be [K]")
    if not (split or plain):
        raise PnpError("nothing to compute")
    if bias_one is not None and K % 8:
        raise PnpError("bias columns need K %% 8 == 0, got K = %d" % K)
    ld3 = 3 * K + (8 if bias_one is not None else 0)
    out3 = torch.empty(x.shape[:-1] + (ld3,), dtype=torch.float16, device=x.device) if split else None
    out1 = torch.empty_like(x) if plain else None
    check(_lib.load().pnp_layernorm_fp16_split3(_p(x), _p(residual), float(residual_scale), _p(residual_bias),
                                                _p(x if residual is not None else None), _p(gamma), _p(beta), float(eps), float(hi_scale),
                                                _p(out3), ld3, float(bias_one or 0.0), _p(out1), _p(flag), M, K, _stream()),
          "pnp_layernorm_fp16_split3")
    return out3, out1


def attention_fp16x3(qkv, in_scale=1.0, softmax_scale=None, flag=None, split_hi_scale=None):
    """softmax(Q K^T * softmax_scale) V for qkv [B,L,3,H,64] fp32 (each value times 1/in_scale) -> [B,L,H*64] fp32
    (pnp_attention_fp16x3: fp32-grade on the fp16 tensor cores).  split_hi_scale: return instead the fp16 [h*s | l | h] operand
    split of the output ([B,L,3*H*64]), written straight from the accumulators."""
    _req(qkv, torch.float32, "qkv", 5)
    B, L, three, H, D = qkv.shape
    if three != 3 or D != 64:
        raise PnpError("qkv must be [B,L,3,H,64]")
    out = out3 = None
    if split_hi_scale is None:
        out = torch.empty((B, L, H * D), dtype=torch.float32, device=qkv.device)
    else:
        out3 = torch.empty((B, L, 3 * H * D), dtype=torch.float16, device=qkv.device)
    lib = _lib.load()
    ws_bytes = lib.pnp_attention_fp16x3_workspace_bytes(B, L, H, D)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=qkv.device)
    check(lib.pnp_attention_fp16x3(_p(qkv), float(in_scale), float(softmax_scale if softmax_scale is not None else D ** -0.5), _p(out),
                                   _p(out3), float(split_hi_scale or 1.0), _p(ws), ws_bytes, _p(flag), B, L, H, D, _stream()),
          "pnp_attention_fp16x3")
    return out if out3 is None else out3


# ----------------------------------------------------------------------------------------------- (f)
def argmax_channels(maps):
    """maps [B,C,N] -> int32 [B,N]; first max wins, NaN counts as max (DRV:387, DRV:1073)."""
    _req(maps, torch.float32, "maps", 3)
    B, C, N = maps.shape
    labels = torch.empty((B, N), dtype=torch.int32, device=maps.device)
    check(_lib.load().pnp_argmax_channels(_p(maps), _p(labels), B, C, N, _stream()), "pnp_argmax_channels")
    return labels


def confusion_accumulate(labels, gt, n_class, hist, lut=None, pred_out=None, bad_count=None):
    """hist[n*gt + lut[label]] += 1 (DRV:1106-1112); labels int32 [B,N], gt float32 [B,N], hist int64 [n,n] (in place)."""
    _req(labels, torch.int32, "labels", 2)
    _req(gt, torch.float32, "gt", 2)
    _req(hist, torch.int64, "hist", 2)
    B, N = labels.shape
    if tuple(gt.shape) != (B, N) or tuple(hist.shape) != (n_class, n_class):
        raise PnpError("gt/hist shape mismatch")
    stride = 0
    if lut is not None:
        _req(lut, torch.int32, "lut", 2)
        stride = lut.shape[1]
    if pred_out is not None:
        _req(pred_out, torch.float32, "pred_out", 2)
    if bad_count is not None:
        _req(bad_count, torch.int32, "bad_count")
    check(_lib.load().pnp_confusion_accumulate(_p(labels), _p(gt), _p(lut), stride, _p(pred_out), _p(hist), _p(bad_count), B, N,
                                               int(n_class), _stream()), "pnp_confusion_accumulate")
    return hist


def label_map(labels, lut, Q=None):
    """ids[b,n] = lut[b, labels[b,n]] and, with the CRF marginals Q [B,N,Cp] of crf_inference, conf[b,n] = Q[b,n,labels[b,n]]
    (pnp_label_map: the relabel of confusion_accumulate without ground truth).  A label outside [0, lut columns) gives id -1 and
    conf -1.  labels int32 [B,N], lut int32 [B,C'] -> (ids int32 [B,N], conf float32 [B,N] or None)."""
    _req(labels, torch.int32, "labels", 2)
    _req(lut, torch.int32, "lut", 2)
    B, N = labels.shape
    if lut.shape[0] != B or lut.shape[1] < 1:
        raise PnpError("lut must be [B, >=1]")
    Cp = 0
    if Q is not None:
        _req(Q, torch.float32, "Q", 3)
        if tuple(Q.shape[:2]) != (B, N) or Q.shape[2] < lut.shape[1]:
            raise PnpError("Q must be [B,N,Cp] with Cp >= the lut's columns")
        Cp = Q.shape[2]
    ids = torch.empty((B, N), dtype=torch.int32, device=labels.device)
    conf = torch.empty((B, N), dtype=torch.float32, device=labels.device) if Q is not None else None
    if labels.numel() == 0:   # an empty tensor's null data pointer would read as a missing argument to the library
        return ids, conf
    check(_lib.load().pnp_label_map(_p(labels), _p(lut), lut.shape[1], _p(Q), Cp, _p(ids), _p(conf), B, N, _stream()),
          "pnp_label_map")
    return ids, conf
