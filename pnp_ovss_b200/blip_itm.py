"""Random-init stand-in for the patched BLIP ITM-large model (BITM:19-314, MED, VIT) with the reference's
capture protocol, whose block-8 cross-attention softmax is the fused CUDA kernel (a).

The checkpoint (model_large_retrieval_flickr.pth) and LAVIS are not available offline, so weights are
normal(0, 0.02) like MED:727-737 / VIT:261-268 and the architecture is restated from the literals in the
reference: ViT-L/16 (width 1024, depth 24, 16 heads, VIT:511-523) and BERT-base with a cross-attention in every
layer (hidden 768, 12 layers, 12 heads, intermediate 3072, encoder_width 1024), ITM head Linear(768, 2).
All GEMMs are plain torch dense contractions (nn.Linear / matmul / SDPA), as north_star prescribes; only the
cross-attention softmax + capture + GradCAM of the selected block is custom.

Two ways to get GradCAM (both end in pnp_xattn_softmax_bwd_gradcam):
  * trimmed (default, SURVEY 7.4): weights frozen, ViT and BERT layers below the block run under no_grad, the loss is
    differentiated w.r.t. the block's attention probabilities only;
  * reference-style (`full_backward=True`): everything requires grad and loss.backward() runs through the whole
    model like BITM:399-404; the autograd.Function's backward emits dscores and the GradCAM in one pass."""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops


class GradcamCapture:
    """Side channel of FusedXattnSoftmax: which head to capture and where the results go."""

    def __init__(self, head, token_mask):
        self.head = int(head)
        self.token_mask = token_mask  # int64 [B, >=T] (the max_length=500 padded attention_mask, BITM:415-416)
        self.probs = None             # [B,h,T,K]  == get_attention_map()
        self.dprobs = None            # [B,h,T,K]  == get_attn_gradients()
        self.gradcam = None           # [B,T-1,K-1]


class FusedXattnSoftmax(torch.autograd.Function):
    """probs = softmax(scores*scale + key_mask); backward = softmax backward fused with the GradCAM of one head."""

    @staticmethod
    def forward(ctx, scores, key_mask, scale, capture):
        probs = ops.softmax_fwd(scores.contiguous(), key_mask, scale)
        ctx.save_for_backward(probs)
        ctx.scale = scale
        ctx.capture = capture
        if capture is not None:
            capture.probs = probs
        return probs

    @staticmethod
    def backward(ctx, dprobs):
        (probs,) = ctx.saved_tensors
        cap = ctx.capture
        dprobs = dprobs.contiguous()
        dscores, cam = ops.softmax_bwd_gradcam(probs, dprobs, cap.token_mask if cap is not None else None,
                                               cap.head if cap is not None else 0, ctx.scale, need_dscores=True,
                                               need_gradcam=cap is not None)
        if cap is not None:
            cap.dprobs = dprobs
            cap.gradcam = cam
        return dscores, None, None, None


# ------------------------------------------------------------------------------------------------- ViT-L/16
def _tf32_split(t):
    """t = hi + lo with hi exactly representable in TF32 (10 explicit mantissa bits, round to nearest)."""
    hi = ((t.view(torch.int32) + 0x1000) & -0x2000).view(torch.float32)
    return hi, t - hi


def _w3(weight):
    """[N,K] frozen weight -> [N,3K] = [W_hi | W_hi | W_lo]: the right-hand operand of the depth-3K TF32 GEMM whose left
    operand is [x_hi | x_lo | x_hi] (ops.tf32_split3 and its fused producers)."""
    w_hi, w_lo = _tf32_split(weight.detach().contiguous())
    return torch.cat([w_hi, w_hi, w_lo], 1).contiguous()


FP16_OUT_SCALE = 2048.0     # 2^11: the factor a 3xFP16 product carries (see _w16 / _mm16)


FP16_BIAS_ONE = 64.0        # the constant the operand kernels write into the first bias column (see _w16)


def _w16(weight, bias=None):
    """[N,K] frozen weight -> (fp16 [N,3K] = [W_h 2^b | W_h | W_l], 2^a) with W = W_h + W_l 2^-11 (W_h = fp16(W), W_l =
    fp16((W - W_h) 2^11)) and a + b = 11: the right-hand operand of the 3xFP16 GEMM whose left operand is
    [x_h 2^a | x_l | x_h] (ops.fp16_split3 and its fused producers).  b is as large as the largest |W| allows, so a is 0
    (no loss of activation range) unless a weight exceeds 32.

    bias: 8 more columns [bias_h 2^11 / FP16_BIAS_ONE | bias_l | 0 x 6] -> [N,3K+8]; against the operand columns
    [FP16_BIAS_ONE, 1, 0 x 6] (ops.layernorm_fp16_split3(bias_one=...)) the GEMM adds 2^11 * bias by itself."""
    w = weight.detach().contiguous().float()
    wmax = float(w.abs().max())
    b = 11 if wmax == 0 else max(0, min(11, int(math.floor(math.log2(65504.0 / wmax)))))
    w_h = w.half()
    w_l = ((w - w_h.float()) * FP16_OUT_SCALE).half()
    cols = [(w_h.float() * (2.0 ** b)).half(), w_h, w_l]
    if bias is not None:
        bv = bias.detach().float()
        if float(bv.abs().max()) * FP16_OUT_SCALE / FP16_BIAS_ONE > 65000.0:
            raise OverflowError("bias too large for the fp16 bias columns")
        b_h = bv.half()
        b_l = ((bv - b_h.float()) * FP16_OUT_SCALE).half()
        tail = torch.zeros((w.shape[0], 8), dtype=torch.float16, device=w.device)
        tail[:, 0] = (b_h.float() * (FP16_OUT_SCALE / FP16_BIAS_ONE)).half()
        tail[:, 1] = b_l
        cols.append(tail)
    return torch.cat(cols, 1).contiguous(), 2.0 ** (11 - b)


def _mm16(x16, w16):
    """2^11 * (x W^T) at fp32-grade accuracy as ONE fp16 tensor-core GEMM (fp32 accumulate and output) over the tripled
    operands: x_h W_h 2^11 + x_l W_h + x_h W_l, with x = x_h + x_l 2^-11.  The caller takes the 2^11 back (a power of two)."""
    return torch.mm(x16.reshape(-1, x16.shape[-1]), w16.t(), out_dtype=torch.float32).view(*x16.shape[:-1], w16.shape[0])


def _mm3(x3, w3, bias=None):
    """y = x W^T (+ bias) at fp32-grade accuracy on the TF32 tensor cores over the tripled operands (fp32 accumulate; the
    dropped x_lo W_lo term is ~2^-22 relative).  Still plain torch dense contractions (cuBLAS).

    Two launches: the main product x_hi W_hi^T (depth K), then the two correction products accumulated onto it
    in place ([x_lo | x_hi] [W_hi | W_lo]^T, depth 2K, beta = 1).  The tensor core adds into its fp32 accumulator with
    truncation, an error that grows with the depth of ONE accumulation chain: keeping the 2^-11-sized corrections out of
    the main chain leaves rms 4.8e-7 of max|y| at K = 1024 (native SIMT fp32: 1.1e-7; all three products in one depth-3K
    chain: 2.1e-6; plain TF32: 5.7e-5) for 9 % more GEMM time (profiles/experiments/r2_gemm_precision.py)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        K = w3.shape[1] // 3
        x2 = x3.reshape(-1, 3 * K)
        y = F.linear(x2[:, :K], w3[:, :K], bias)
        y.addmm_(x2[:, K:], w3[:, K:].t())
        return y.view(*x3.shape[:-1], w3.shape[0])
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


class _Linear3(torch.autograd.Function):
    """y = x W^T + b for a FROZEN weight on the TF32 tensor cores at fp32 grade (exact hi/lo split, three products), forward and
    backward: dL/dx = dL/dy W is the same kind of product against the split of W^T.  TF32 keeps fp32's exponent range, so the
    tiny gradients of the trimmed backward (1e-6 and below) lose nothing -- which is why the text side does not use fp16."""

    @staticmethod
    def forward(ctx, x, w3, wt3, bias):
        ctx.wt3 = wt3
        ctx.x_shape = x.shape
        y = _mm3(ops.tf32_split3(x.reshape(-1, x.shape[-1]).contiguous()), w3, bias)
        return y.view(*x.shape[:-1], w3.shape[0])

    @staticmethod
    def backward(ctx, gy):
        gx = _mm3(ops.tf32_split3(gy.reshape(-1, gy.shape[-1]).contiguous()), ctx.wt3)
        return gx.view(ctx.x_shape), None, None, None


def _plain_linear(module, x):
    return module(x)


class _VitBlock(nn.Module):
    def __init__(self, dim, heads, mlp_ratio=4.0):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.qkv = nn.Linear(dim, dim * 3)
        self.proj = nn.Linear(dim, dim)
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.fc1 = nn.Linear(dim, int(dim * mlp_ratio))
        self.fc2 = nn.Linear(int(dim * mlp_ratio), dim)
        self.heads = heads

    def forward(self, x):
        B, L, D = x.shape
        qkv = self.qkv(self.norm1(x)).view(B, L, 3, self.heads, D // self.heads).permute(2, 0, 3, 1, 4)
        a = F.scaled_dot_product_attention(qkv[0], qkv[1], qkv[2])
        x = x + self.proj(a.transpose(1, 2).reshape(B, L, D))
        return x + self.fc2(F.gelu(self.fc1(self.norm2(x))))


class VisionTransformer(nn.Module):
    def __init__(self, img_size=336, patch=16, dim=1024, depth=24, heads=16):
        super().__init__()
        self.patch_embed = nn.Conv2d(3, dim, patch, patch)
        n = (img_size // patch) ** 2
        self.cls_token = nn.Parameter(torch.zeros(1, 1, dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, n + 1, dim))
        self.blocks = nn.ModuleList([_VitBlock(dim, heads) for _ in range(depth)])
        self.norm = nn.LayerNorm(dim, eps=1e-6)

    def forward(self, x):
        x = self.patch_embed(x).flatten(2).transpose(1, 2)
        x = torch.cat([self.cls_token.expand(x.shape[0], -1, -1), x], 1) + self.pos_embed
        for blk in self.blocks:
            x = blk(x)
        return self.norm(x)


# ------------------------------------------------------------------------------------------------- BERT with cross-attention
class CrossAttentionSelf(nn.Module):
    """BertSelfAttention(is_cross_attention=True), MED:126-311, with the capture protocol of MED:164-180."""

    def __init__(self, hidden, heads, enc_width):
        super().__init__()
        self.query = nn.Linear(hidden, hidden)
        self.key = nn.Linear(enc_width, hidden)
        self.value = nn.Linear(enc_width, hidden)
        self.heads = heads
        self.save_attention = False
        self.capture = None          # GradcamCapture while save_attention is on
        self.detach_probs = False    # trimmed mode: probs become the leaf the loss is differentiated against

    def get_attention_map(self):
        return self.capture.probs

    def get_attn_gradients(self):
        return self.capture.dprobs

    def _split(self, x):
        B, L, D = x.shape
        return x.view(B, L, self.heads, D // self.heads).permute(0, 2, 1, 3)

    def forward(self, hidden, enc, enc_mask=None, kv=None, lin=_plain_linear):
        """kv: (key(enc), value(enc), s) precomputed for all blocks in one tensor-core GEMM, both [B,L,hidden] and both carrying
        the power-of-two factor s (1, or 2^11 in the 3xFP16 form), which the score scale and the context take back exactly."""
        k, v, kv_s = kv if kv is not None else (self.key(enc), self.value(enc), 1.0)
        q, k, v = self._split(lin(self.query, hidden)), self._split(k), self._split(v)
        scores = torch.matmul(q, k.transpose(-1, -2))                       # MED:228
        scale = 1.0 / math.sqrt(q.shape[-1]) / kv_s                          # MED:267
        if self.save_attention:
            probs = FusedXattnSoftmax.apply(scores, enc_mask, scale, self.capture)   # MED:269-283 fused
            if self.detach_probs:
                probs = probs.detach().requires_grad_(True)
                self.capture.probs = probs
        else:
            s = scores * scale
            if enc_mask is not None:
                s = s + enc_mask[:, None, None, :]
            probs = torch.softmax(s, -1)
        ctx = torch.matmul(probs, v)                                         # MED:300
        if kv_s != 1.0:
            ctx = ctx * (1.0 / kv_s)
        B, h, T, d = ctx.shape
        return ctx.permute(0, 2, 1, 3).reshape(B, T, h * d)


class _BertLayer(nn.Module):
    def __init__(self, hidden, heads, inter, enc_width, eps=1e-12):
        super().__init__()
        self.heads = heads
        self.q, self.k, self.v = nn.Linear(hidden, hidden), nn.Linear(hidden, hidden), nn.Linear(hidden, hidden)
        self.attn_out = nn.Linear(hidden, hidden)
        self.attn_ln = nn.LayerNorm(hidden, eps=eps)
        self.crossattention = nn.Module()
        self.crossattention.self = CrossAttentionSelf(hidden, heads, enc_width)
        self.cross_out = nn.Linear(hidden, hidden)
        self.cross_ln = nn.LayerNorm(hidden, eps=eps)
        self.inter = nn.Linear(hidden, inter)
        self.out = nn.Linear(inter, hidden)
        self.out_ln = nn.LayerNorm(hidden, eps=eps)

    def self_attention(self, x, add_mask, lin=_plain_linear):
        B, T, D = x.shape
        sp = lambda t: t.view(B, T, self.heads, D // self.heads).permute(0, 2, 1, 3)
        a = F.scaled_dot_product_attention(sp(lin(self.q, x)), sp(lin(self.k, x)), sp(lin(self.v, x)), attn_mask=add_mask)
        return self.attn_ln(lin(self.attn_out, a.permute(0, 2, 1, 3).reshape(B, T, D)) + x)

    def cross_and_ffn(self, x, enc, kv=None, lin=_plain_linear):
        x = self.cross_ln(lin(self.cross_out, self.crossattention.self(x, enc, kv=kv, lin=lin)) + x)
        return self.out_ln(lin(self.out, F.gelu(lin(self.inter, x))) + x)


class _TextEncoderView:
    """The slice of the LAVIS XBertEncoder surface the reference touches: `.base_model` (itself) and `.encoder.layer`."""

    def __init__(self, model):
        self.encoder = self
        self.layer = model.layer

    @property
    def base_model(self):
        return self


class BlipITM(nn.Module):
    def __init__(self, img_size=336, tokenizer=None, vocab=30524, hidden=768, layers=12, heads=12, inter=3072,
                 vit_dim=1024, vit_depth=24, vit_heads=16, max_pos=512):
        super().__init__()
        self.tokenizer = tokenizer
        self.patch_num = img_size // 16
        self.visual_encoder = VisionTransformer(img_size, 16, vit_dim, vit_depth, vit_heads)
        self.word_emb = nn.Embedding(vocab, hidden)
        self.pos_emb = nn.Embedding(max_pos, hidden)
        self.emb_ln = nn.LayerNorm(hidden, eps=1e-12)
        self.layer = nn.ModuleList([_BertLayer(hidden, heads, inter, vit_dim) for _ in range(layers)])
        self.itm_head = nn.Linear(hidden, 2)
        self.apply(self._init)
        nn.init.normal_(self.visual_encoder.pos_embed, std=0.02)
        nn.init.normal_(self.visual_encoder.cls_token, std=0.02)
        self.gemm_precision = "fp32"

    @staticmethod
    def _init(m):
        if isinstance(m, (nn.Linear, nn.Embedding, nn.Conv2d)):
            nn.init.normal_(m.weight, mean=0.0, std=0.02)
            if getattr(m, "bias", None) is not None:
                nn.init.zeros_(m.bias)
        elif isinstance(m, nn.LayerNorm):
            nn.init.ones_(m.weight)
            nn.init.zeros_(m.bias)

    _CACHES = ("_w3_cache", "_text3_cache", "_text_graphs", "_text_graph_stamp", "_vit_graphs", "_kv_buffers", "_fp16_flags")

    def __deepcopy__(self, memo):
        """Copies the module without its derived state (weight splits, K/V buffers, captured CUDA graphs): all of it is rebuilt
        on first use, and a CUDA graph cannot be copied."""
        import copy
        saved = {k: self.__dict__.pop(k) for k in self._CACHES if k in self.__dict__}
        try:
            new = self.__class__.__new__(self.__class__)
            memo[id(self)] = new
            new.__dict__ = copy.deepcopy(self.__dict__, memo)
            return new
        finally:
            self.__dict__.update(saved)

    # ---- the reference's attribute path / checkpoint ---------------------------------------------------
    @property
    def text_encoder(self):
        """model.text_encoder.base_model.base_model.encoder.layer[i].crossattention.self (BITM:388-392) resolves to
        this model's cross-attention modules."""
        return _TextEncoderView(self)

    def load_lavis_checkpoint(self, path_or_state_dict):
        """Weights of the reference's LAVIS BlipITM (YAML:10) -> this model; see lavis_compat.load_lavis_state_dict."""
        from .lavis_compat import load_lavis_state_dict
        sd = path_or_state_dict
        if not isinstance(sd, dict):
            sd = torch.load(sd, map_location="cpu")
        return load_lavis_state_dict(self, sd)

    # ---- pieces -----------------------------------------------------------------------------------
    def _tokenize(self, text_input, device):
        text = self.tokenizer(text_input, padding="longest", truncation=True, max_length=500, return_tensors="pt")  # BITM:230-236
        ids = text.input_ids.to(device).clone()
        ids[:, 0] = self.tokenizer.enc_token_id  # BITM:238-239
        return ids, text.attention_mask.to(device)

    def _embed(self, ids):
        pos = torch.arange(ids.shape[1], device=ids.device)
        return self.emb_ln(self.word_emb(ids) + self.pos_emb(pos)[None])

    def _vit(self, imgs):
        if self.gemm_precision == "bf16":
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return self.visual_encoder(imgs).float()
        return self.visual_encoder(imgs)

    # ---- "3xtf32" / "3xfp16": the frozen-weight encoder pass with every large GEMM on the tensor cores at fp32-grade accuracy
    SPLIT_MODES = ("3xtf32", "3xfp16")

    def _weights3(self, mode="3xtf32"):
        """Tripled splits of the frozen weights for `mode` ([W_hi | W_hi | W_lo] fp32, see _w3; or fp16 with its activation
        scale, see _w16), rebuilt when a parameter changes."""
        ve = self.visual_encoder
        params = [ve.patch_embed.weight] + [p for blk in ve.blocks for p in (blk.qkv.weight, blk.proj.weight, blk.fc1.weight, blk.fc2.weight)]
        params += [p for lyr in self.layer for p in (lyr.crossattention.self.key.weight, lyr.crossattention.self.value.weight)]
        stamp = tuple((p.data_ptr(), p._version) for p in params)
        caches = self.__dict__.setdefault("_w3_cache", {})
        cache = caches.get(mode)
        if cache is None or cache["stamp"] != stamp:
            half = mode == "3xfp16"
            prep = (lambda w, b=None: _w16(w, b)) if half else (lambda w, b=None: (_w3(w), 1.0))
            with torch.no_grad():
                xs = [lyr.crossattention.self for lyr in self.layer]
                kv_bias = torch.cat([b for x in xs for b in (x.key.bias, x.value.bias)], 0).contiguous()
                cache = {
                    "stamp": stamp,
                    "patch": prep(ve.patch_embed.weight.reshape(ve.patch_embed.weight.shape[0], -1)),
                    # (qkv with its bias folded into the operand in the fp16 form, proj, fc1, fc2)
                    "blocks": [(prep(blk.qkv.weight, blk.qkv.bias), prep(blk.proj.weight), prep(blk.fc1.weight), prep(blk.fc2.weight))
                               for blk in ve.blocks],
                    # key/value projections of all cross-attention blocks as one [layers*2*hidden, 3*enc_width (+8)] operand
                    "kv": prep(torch.cat([w for x in xs for w in (x.key.weight, x.value.weight)], 0), kv_bias),
                    "kv_bias": kv_bias,
                }
            caches[mode] = cache
        return cache

    def _text_linear(self):
        """lin(module, x) for the text side: in the tensor-core modes (frozen weights, CUDA) every nn.Linear of the BERT layers
        runs through _Linear3 (forward and backward on the TF32 tensor cores at fp32 grade); plain module call otherwise."""
        if self.gemm_precision not in self.SPLIT_MODES or any(p.requires_grad for p in self.layer.parameters()):
            return _plain_linear
        cache = self.__dict__.setdefault("_text3_cache", {})

        def lin(module, x):
            if not x.is_cuda or module.in_features % 4 or module.out_features % 4:
                return module(x)
            w = module.weight
            ent = cache.get(id(module))
            if ent is None or ent[0] != (w.data_ptr(), w._version):
                with torch.no_grad():
                    ent = ((w.data_ptr(), w._version), _w3(w), _w3(w.t().contiguous()))
                cache[id(module)] = ent
            return _Linear3.apply(x, ent[1], ent[2], module.bias)

        return lin

    def fp16_overflow_flag(self, device):
        """Device int32 raised by the 3xFP16 operand kernels when an activation does not fit fp16; read it once per run
        (`check_fp16_overflow`), not per pass."""
        flags = self.__dict__.setdefault("_fp16_flags", {})
        key = str(device)
        if key not in flags:
            flags[key] = torch.zeros(1, dtype=torch.int32, device=device)
        return flags[key]

    def check_fp16_overflow(self):
        for flag in self.__dict__.get("_fp16_flags", {}).values():
            if int(flag.item()):
                raise ops.PnpError("an activation left fp16's range in a 3xFP16 GEMM operand: use gemm_precision='3xtf32' for this model")

    def _vit3(self, imgs, want_plain=False, mode="3xtf32"):
        """ViT-L forward (VIT:274-290) under no_grad with the GEMM operands prepared by the fused split kernels:
        residual add + LayerNorm + split, GELU + split, plain split.  Returns (enc3 [B,L,3D] split, enc [B,L,D] or None).
        mode "3xfp16": the products carry a factor 2^11 that the next fused kernel takes back (inv)."""
        ve = self.visual_encoder
        w = self._weights3(mode)
        half = mode == "3xfp16"
        inv = 1.0 / FP16_OUT_SCALE if half else 1.0
        flag = self.fp16_overflow_flag(imgs.device) if half else None
        mm = _mm16 if half else _mm3

        def split(x, in_scale, wt):
            return ops.fp16_split3(x, in_scale, wt[1], flag) if half else ops.tf32_split3(x)

        def ln(x, norm, wt, r=None, rb=None, fold_bias=False, **kw):
            if half:
                return ops.layernorm_fp16_split3(x, norm.weight, norm.bias, norm.eps, residual=r, residual_scale=inv, residual_bias=rb,
                                                 hi_scale=wt[1], flag=flag, bias_one=FP16_BIAS_ONE if fold_bias else None, **kw)
            return ops.layernorm_tf32_split3(x, norm.weight, norm.bias, norm.eps, residual=r, residual_bias=rb, **kw)

        B, _, S, _ = imgs.shape
        ps = ve.patch_embed.kernel_size[0]
        G = S // ps
        D = ve.pos_embed.shape[-1]
        patches = imgs.view(B, 3, G, ps, G, ps).permute(0, 2, 4, 1, 3, 5).reshape(B * G * G, 3 * ps * ps).contiguous()
        pe = torch.add(ve.patch_embed.bias, mm(split(patches, 1.0, w["patch"]), w["patch"][0]), alpha=inv).view(B, G * G, D)
        x = (torch.cat([ve.cls_token.expand(B, -1, -1), pe], 1) + ve.pos_embed).contiguous()
        L = x.shape[1]
        r = rb = None
        for blk, (w_qkv, w_proj, w_fc1, w_fc2) in zip(ve.blocks, w["blocks"]):
            h3, _ = ln(x, blk.norm1, w_qkv, r, rb, fold_bias=True)
            # fp16 form: the GEMM adds the bias itself (operand columns) and q, k, v come out times 2^11 -- a power of two that
            # the attention's scale (2^-22 / sqrt(d)) and the next split (2^-11) take back exactly
            qkv = mm(h3, w_qkv[0]) if half else _mm3(h3, w_qkv[0], blk.qkv.bias)
            hd = D // blk.heads
            if half and hd == 64:
                # the attention itself on the fp16 tensor cores with the same hi/lo split (pnp_attention_fp16x3): unscaled output
                a3 = ops.attention_fp16x3(qkv.view(B, L, 3, blk.heads, hd), inv, 1.0 / math.sqrt(hd), flag, split_hi_scale=w_proj[1])
                r = mm(a3, w_proj[0])
            else:
                qkv = qkv.view(B, L, 3, blk.heads, hd).permute(2, 0, 3, 1, 4)
                a = F.scaled_dot_product_attention(qkv[0], qkv[1], qkv[2], scale=inv * inv / math.sqrt(hd))
                r = mm(split(a.transpose(1, 2).reshape(B, L, D).contiguous(), inv, w_proj), w_proj[0])
            h3, _ = ln(x, blk.norm2, w_fc1, r, blk.proj.bias)
            f = mm(h3, w_fc1[0])
            g3 = (ops.gelu_fp16_split3(f, blk.fc1.bias, inv, w_fc2[1], flag) if half else ops.gelu_tf32_split3(f, blk.fc1.bias))
            r, rb = mm(g3, w_fc2[0]), blk.fc2.bias
        return ln(x, ve.norm, w["kv"], r, rb, fold_bias=True, split=True, plain=want_plain)

    def _cross_kv3(self, enc3, mode="3xtf32"):
        """key(enc) / value(enc) of every cross-attention block (MED:201-221) in one GEMM -> list of (k, v, s) with k, v
        [B,L,hidden] carrying the factor s (2^11 in the fp16 form: the cross-attention takes it back, see CrossAttentionSelf)."""
        w = self._weights3(mode)
        n = len(self.layer)
        half = mode == "3xfp16"
        # One persistent output buffer per shape: the text-pass CUDA graph reads K/V at fixed addresses, so the GEMM writes there
        # directly and nothing is copied.  (Passes on one stream are ordered; a pass never outlives the next one's GEMM.)
        bufs = self.__dict__.setdefault("_kv_buffers", {})
        M, N = enc3.shape[0] * enc3.shape[1], w["kv"][0].shape[0]
        key = (M, N, str(enc3.device))
        if key not in bufs:
            bufs[key] = torch.empty((M, N), dtype=torch.float32, device=enc3.device)
        out = bufs[key]
        x2 = enc3.reshape(M, enc3.shape[-1])
        if half:
            torch.mm(x2, w["kv"][0].t(), out_dtype=torch.float32, out=out)
        else:
            prev = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = True
            try:
                K = w["kv"][0].shape[1] // 3
                torch.addmm(w["kv_bias"], x2[:, :K], w["kv"][0][:, :K].t(), out=out)
                out.addmm_(x2[:, K:], w["kv"][0][:, K:].t())
            finally:
                torch.backends.cuda.matmul.allow_tf32 = prev
        kv = out.view(enc3.shape[0], enc3.shape[1], n, 2, -1)
        s = FP16_OUT_SCALE if half else 1.0
        return [(kv[:, :, i, 0], kv[:, :, i, 1], s) for i in range(n)]

    USE_VIT_GRAPH = True

    def _encode(self, imgs):
        """(enc or None, per-block cross-attention (k, v) or [None]*n) for the current gemm_precision."""
        mode = self.gemm_precision
        if mode in self.SPLIT_MODES and imgs.is_cuda and not any(p.requires_grad for p in self.visual_encoder.parameters()):
            with torch.no_grad():
                if self.USE_VIT_GRAPH:
                    kvs = self._encode_graphed(imgs, mode)
                    if kvs is not None:
                        return None, kvs
                enc3, _ = self._vit3(imgs, mode=mode)
                return None, self._cross_kv3(enc3, mode)
        return self._vit(imgs), [None] * len(self.layer)

    def _encode_graphed(self, imgs, mode):
        """The encoder pass + the K/V GEMM replayed from a CUDA graph (one per image shape): ~330 launches whose host-side issue
        otherwise leaves the GPU idle for ~3 ms per pass.  The graph's only output is the persistent K/V buffer of _cross_kv3.
        Returns None when capture is impossible here."""
        graphs = self.__dict__.setdefault("_vit_graphs", {})
        self._weights3(mode)                       # (re)builds the splits when a weight changed ...
        stamp = self.__dict__["_w3_cache"][mode]["stamp"]
        key = (tuple(imgs.shape), str(imgs.device), mode)
        ent = graphs.get(key)
        if ent is not None and ent is not False and ent[2] != stamp:
            ent = None                             # ... and a graph captured with the old splits is dropped
        if ent is False:
            return None
        if ent is None:
            static = imgs.clone()
            try:
                cur = torch.cuda.current_stream()
                side = torch.cuda.Stream()
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    for _ in range(2):
                        self._cross_kv3(self._vit3(static, mode=mode)[0], mode)
                cur.wait_stream(side)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    kvs = self._cross_kv3(self._vit3(static, mode=mode)[0], mode)
                ent = (g, static, stamp, kvs)
            except Exception as e:  # noqa: BLE001 -- eager is always correct
                import warnings
                warnings.warn("encoder CUDA graph capture failed (%s); running it eagerly" % str(e).splitlines()[0][:200])
                torch.cuda.synchronize()
                graphs[key] = False
                return None
            graphs[key] = ent
        g, static, _, kvs = ent
        static.copy_(imgs)
        g.replay()
        return kvs

    def forward(self, visual_input, text_input=None, match_head="itm"):
        """ITM logits [B,2] (BITM:217-249, match_head='itm').  Also takes the LAVIS call form
        model({"image": ..., "text_input": ...}, match_head="itm") of BITM:395."""
        if isinstance(visual_input, dict):
            visual_input, text_input = visual_input["image"], visual_input["text_input"]
        if match_head != "itm":
            raise NotImplementedError("only the ITM head is on the mask-extraction path")
        ids, att = self._tokenize(text_input, visual_input.device)
        enc, kvs = self._encode(visual_input)
        add_mask = ((1.0 - att.float()) * -10000.0)[:, None, None, :]
        lin = self._text_linear()
        x = self._embed(ids)
        for lyr, kv in zip(self.layer, kvs):
            x = lyr.cross_and_ffn(lyr.self_attention(x, add_mask, lin), enc, kv, lin)
        return self.itm_head(x[:, 0])

    def _text_pass(self, ids, add_mask, token_mask, enc, kvs, layer, head, cap):
        """The text side of the trimmed GradCAM pass: BERT layers below `layer` without grad, the block's attention
        probabilities as the leaf, the loss differentiated w.r.t. them, the fused GradCAM kernel.  -> (cam [B,T-1,K-1], logits)."""
        lin = self._text_linear()
        with torch.no_grad():
            x = self._embed(ids)
            for lyr, kv in zip(self.layer[:layer], kvs):
                x = lyr.cross_and_ffn(lyr.self_attention(x, add_mask, lin), enc, kv, lin)
            x = self.layer[layer].self_attention(x, add_mask, lin)
        with torch.enable_grad():
            x = self.layer[layer].cross_and_ffn(x, enc, kvs[layer], lin)   # probs become a leaf inside (detach_probs)
            for lyr, kv in zip(self.layer[layer + 1:], kvs[layer + 1:]):
                x = lyr.cross_and_ffn(lyr.self_attention(x, add_mask, lin), enc, kv, lin)
            out = self.itm_head(x[:, 0])
            loss = out[:, 1].sum()
            (dprobs,) = torch.autograd.grad(loss, cap.probs)
        cap.dprobs = dprobs
        _, cam = ops.softmax_bwd_gradcam(cap.probs.detach(), dprobs.contiguous(), token_mask, head,
                                         1.0 / math.sqrt(64), need_dscores=False, need_gradcam=True)
        return cam, out.detach()

    # ---- the text pass as a CUDA graph -----------------------------------------------------------------
    USE_TEXT_GRAPH = True

    def _text_pass_graphed(self, ids, add_mask, token_mask, kvs, layer, head):
        """_text_pass replayed from a CUDA graph: the text side is ~700 launches of kernels that each run for microseconds
        (B*T = 875 rows at cfg1), so issued one by one it is bound by launch latency, not by the GPU.  One graph per
        (shapes, block, head); inputs are copied into the graph's static buffers, the result is copied out.
        Returns None when capture is impossible here (the caller then runs the eager pass)."""
        graphs = self.__dict__.setdefault("_text_graphs", {})
        stamp = tuple(p._version for p in self.layer.parameters()) + tuple(p._version for p in self.itm_head.parameters())
        if self.__dict__.get("_text_graph_stamp") != stamp:     # a graph holds the addresses of the weight splits it was captured with
            graphs.clear()
            self.__dict__["_text_graph_stamp"] = stamp
        k0, v0, s0 = kvs[0]
        key = (tuple(ids.shape), tuple(k0.shape), k0.data_ptr(), int(layer), int(head), float(s0), str(ids.device), token_mask.shape[1],
               self.gemm_precision)
        ent = graphs.get(key)
        if ent is False:
            return None
        if ent is None:
            st = {"ids": ids.clone(), "add_mask": add_mask.clone(), "token_mask": token_mask.clone()}
            skvs = kvs                             # views of the persistent K/V buffer of _cross_kv3: fixed addresses
            xattn = self.layer[layer].crossattention.self

            def run():
                cap = GradcamCapture(head, st["token_mask"])
                xattn.save_attention, xattn.capture, xattn.detach_probs = True, cap, True
                try:
                    return self._text_pass(st["ids"], st["add_mask"], st["token_mask"], None, skvs, layer, head, cap)
                finally:
                    xattn.save_attention, xattn.capture, xattn.detach_probs = False, None, False

            try:
                cur = torch.cuda.current_stream()
                side = torch.cuda.Stream()
                side.wait_stream(cur)
                with torch.cuda.stream(side):      # warm-up off the capture stream (autograd buffers, cuBLAS workspaces)
                    for _ in range(2):
                        run()
                cur.wait_stream(side)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    st["cam"], st["out"] = run()
                ent = (g, st)
            except Exception as e:  # noqa: BLE001 -- a failed capture must not take the pass down; eager is always correct
                import warnings
                warnings.warn("text-pass CUDA graph capture failed (%s); running it eagerly" % str(e).splitlines()[0][:200])
                torch.cuda.synchronize()
                graphs[key] = False
                return None
            graphs[key] = ent
        g, st = ent
        st["ids"].copy_(ids)
        st["add_mask"].copy_(add_mask)
        st["token_mask"].copy_(token_mask)
        g.replay()
        return st["cam"].clone(), st["out"].clone()

    # ---- GradCAM of one (block, head) ----------------------------------------------------------------
    def gradcam(self, visual_input, text_input, tokenized_text, layer=7, head=9, full_backward=False):
        """Returns (gradcam [B,T-1,P,P], itm_logits [B,2]) for block `layer`, head `head` (BITM:386-457)."""
        dev = visual_input.device
        ids, att = self._tokenize(text_input, dev)
        B, T = ids.shape
        token_mask = tokenized_text.attention_mask.to(dev)
        if token_mask.dtype != torch.int64:
            token_mask = token_mask.long()
        token_mask = token_mask.contiguous()
        cap = GradcamCapture(head, token_mask)
        xattn = self.layer[layer].crossattention.self
        xattn.save_attention, xattn.capture, xattn.detach_probs = True, cap, not full_backward
        add_mask = ((1.0 - att.float()) * -10000.0)[:, None, None, :]
        try:
            if full_backward:
                with torch.enable_grad():
                    enc = self._vit(visual_input)
                    x = self._embed(ids)
                    for lyr in self.layer:
                        x = lyr.cross_and_ffn(lyr.self_attention(x, add_mask), enc)
                    out = self.itm_head(x[:, 0])
                    loss = out[:, 1].sum()       # BITM:399
                    self.zero_grad()
                    loss.backward()              # BITM:404; FusedXattnSoftmax.backward fills cap.gradcam
                cam = cap.gradcam
            else:
                with torch.no_grad():
                    enc, kvs = self._encode(visual_input)
                res = None
                if self.USE_TEXT_GRAPH and enc is None and self._text_linear() is not _plain_linear:
                    res = self._text_pass_graphed(ids, add_mask, token_mask, kvs, layer, head)
                cam, out = res if res is not None else self._text_pass(ids, add_mask, token_mask, enc, kvs, layer, head, cap)
        finally:
            xattn.save_attention, xattn.capture, xattn.detach_probs = False, None, False
        P = self.patch_num
        return cam.view(B, T - 1, P, P), out.detach()
