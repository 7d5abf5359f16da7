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
import types

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


def _mm16(x16, w16, out=None):
    """2^11 * (x W^T) at fp32-grade accuracy as ONE fp16 tensor-core GEMM (fp32 accumulate and output) over the tripled
    operands: x_h W_h 2^11 + x_l W_h + x_h W_l, with x = x_h + x_l 2^-11.  The caller takes the 2^11 back (a power of two)."""
    y = torch.mm(x16.reshape(-1, x16.shape[-1]), w16.t(), out_dtype=torch.float32, out=out)
    return y.view(*x16.shape[:-1], w16.shape[0])


def _mm3(x3, w3, bias=None, out=None):
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
        xh, wh = x2[:, :K], w3[:, :K].t()
        y = torch.mm(xh, wh, out=out) if bias is None else torch.addmm(bias, xh, wh, out=out)   # = F.linear on 2-D operands
        y.addmm_(x2[:, K:], w3[:, K:].t())
        return y.view(*x3.shape[:-1], w3.shape[0])
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


# The two operand forms of the split GEMM modes.  `prep(W, b)` makes the right-hand operand (weight, hi_scale, b) of a frozen
# weight; `split` / `ln` / `gelu` write the matching left-hand operand of an activation (the fp16 forms raise `flag` when a
# value leaves fp16's range); `mm` multiplies the two, and the product carries the factor `scale`, which the next producer
# takes back exactly (a power of two).
#   3xtf32: [hi | lo | hi] fp32, two launches (_mm3), the bias added by the GEMM from the live parameter, scale 1.
#   3xfp16: [h 2^a | l | h] fp16, one launch (_mm16), scale 2^11; a bias is folded into 8 more weight columns (_w16), and `ln`
#           writes the matching [FP16_BIAS_ONE, 1, 0 x 6] columns for an operand that carries one.
_FORMS = {
    "3xtf32": types.SimpleNamespace(
        scale=1.0,
        prep=lambda w, b=None: (_w3(w), 1.0, b),
        mm=lambda x3, op, out=None: _mm3(x3, op[0], op[2], out),
        split=lambda x, in_scale, op, flag: ops.tf32_split3(x),
        ln=lambda x, norm, op, flag, r=None, rb=None, **kw: ops.layernorm_tf32_split3(
            x, norm.weight, norm.bias, norm.eps, residual=r, residual_bias=rb, **kw),
        gelu=lambda x, bias, op, flag: ops.gelu_tf32_split3(x, bias)),
    "3xfp16": types.SimpleNamespace(
        scale=FP16_OUT_SCALE,
        prep=lambda w, b=None: _w16(w, b) + (b,),
        mm=lambda x16, op, out=None: _mm16(x16, op[0], out),
        split=lambda x, in_scale, op, flag: ops.fp16_split3(x, in_scale, op[1], flag),
        ln=lambda x, norm, op, flag, r=None, rb=None, **kw: ops.layernorm_fp16_split3(
            x, norm.weight, norm.bias, norm.eps, residual=r, residual_scale=1.0 / FP16_OUT_SCALE, residual_bias=rb, hi_scale=op[1],
            flag=flag, bias_one=None if op[2] is None else FP16_BIAS_ONE, **kw),
        gelu=lambda x, bias, op, flag: ops.gelu_fp16_split3(x, bias, 1.0 / FP16_OUT_SCALE, op[1], flag)),
}


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

    def __deepcopy__(self, memo):
        """Copies the module without its derived state (see _refresh; rebuilt on first use, and a CUDA graph cannot be copied)
        and with clear fp16 overflow flags."""
        import copy
        saved = {k: self.__dict__.pop(k) for k in ("_derived", "_fp16_flags") if k in self.__dict__}
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
        """Weights of the reference's LAVIS BlipITM (YAML:10) -> this model, with clear fp16 overflow flags; see
        lavis_compat.load_lavis_state_dict."""
        from .lavis_compat import load_lavis_state_dict
        sd = path_or_state_dict
        if not isinstance(sd, dict):
            sd = torch.load(sd, map_location="cpu")
        ignored = load_lavis_state_dict(self, sd)
        for flag in self.__dict__.get("_fp16_flags", {}).values():
            flag.zero_()
        return ignored

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

    def _refresh(self):
        """Everything derived from the parameters -- weight operands per split mode, text-side _Linear3 splits, the K/V output
        buffers and the captured CUDA graphs, which hold the addresses of all of these -- lives in one dict that is dropped
        when the stamp of the parameters changes.  The stamp is (data_ptr, _version) of every weight and bias: it sees in-place
        edits (load_state_dict copies in place) and moves (.to()).  Called once per forward() / gradcam() of a split mode
        (_encode).  -> True when no parameter requires grad (the split paths serve frozen weights only)."""
        stamp, grad, mods = [], False, [self]
        for m in mods:
            mods.extend(m._modules.values())
            for p in m._parameters.values():
                stamp.append((p.data_ptr(), p._version))
                grad = grad or p.requires_grad
        if self.__dict__.get("_derived", {}).get("stamp") != stamp:
            self.__dict__["_derived"] = {"stamp": stamp, "weights": {}, "text": {}, "kv": {}, "graphs": {}}
        return not grad

    def _cache(self, name):
        """One part of the derived state of the current parameters (see _refresh)."""
        if "_derived" not in self.__dict__:
            self._refresh()
        return self.__dict__["_derived"][name]

    def _weights3(self, mode="3xtf32"):
        """Operands of the frozen encoder weights in `mode`'s form (see _FORMS)."""
        cache = self._cache("weights")
        if mode not in cache:
            prep = _FORMS[mode].prep
            ve = self.visual_encoder
            xs = [lyr.crossattention.self for lyr in self.layer]
            with torch.no_grad():
                cache[mode] = {
                    "patch": prep(ve.patch_embed.weight.reshape(ve.patch_embed.weight.shape[0], -1)),
                    "blocks": [(prep(blk.qkv.weight, blk.qkv.bias), prep(blk.proj.weight), prep(blk.fc1.weight), prep(blk.fc2.weight))
                               for blk in ve.blocks],
                    # key/value projections of all cross-attention blocks as one [layers*2*hidden, 3*enc_width (+8)] operand
                    "kv": prep(torch.cat([w for x in xs for w in (x.key.weight, x.value.weight)], 0),
                               torch.cat([b for x in xs for b in (x.key.bias, x.value.bias)], 0).contiguous()),
                }
        return cache[mode]

    def _linear3(self, module, x):
        """lin(module, x) of the text side on the split path: an nn.Linear of the BERT layers through _Linear3 (forward and
        backward on the TF32 tensor cores at fp32 grade)."""
        if module.in_features % 4 or module.out_features % 4:
            return module(x)
        cache = self._cache("text")
        if module not in cache:
            with torch.no_grad():
                cache[module] = (_w3(module.weight), _w3(module.weight.t().contiguous()))
        return _Linear3.apply(x, *cache[module], module.bias)

    def fp16_overflow_flag(self, device):
        """Device int32 raised by the 3xFP16 operand kernels when an activation does not fit fp16; read it once per run
        (`check_fp16_overflow`), not per pass.  Not part of the derived state (_refresh): captured graphs hold its address, and
        an overflow seen before a weight change is still reported."""
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
        Every product carries the factor of `mode`'s form (2^11 in 3xfp16), which the next fused kernel takes back (inv)."""
        ve = self.visual_encoder
        f, w = _FORMS[mode], self._weights3(mode)
        inv = 1.0 / f.scale
        flag = self.fp16_overflow_flag(imgs.device)
        B, _, S, _ = imgs.shape
        ps = ve.patch_embed.kernel_size[0]
        G = S // ps
        D = ve.pos_embed.shape[-1]
        patches = imgs.view(B, 3, G, ps, G, ps).permute(0, 2, 4, 1, 3, 5).reshape(B * G * G, 3 * ps * ps).contiguous()
        pe = torch.add(ve.patch_embed.bias, f.mm(f.split(patches, 1.0, w["patch"], flag), w["patch"]), alpha=inv).view(B, G * G, D)
        x = (torch.cat([ve.cls_token.expand(B, -1, -1), pe], 1) + ve.pos_embed).contiguous()
        L = x.shape[1]
        r = rb = None
        for blk, (w_qkv, w_proj, w_fc1, w_fc2) in zip(ve.blocks, w["blocks"]):
            # q, k, v come out times the form's factor -- a power of two that the attention's scale and the next split take back
            qkv = f.mm(f.ln(x, blk.norm1, w_qkv, flag, r, rb)[0], w_qkv)
            hd = D // blk.heads
            if mode == "3xfp16" and hd == 64:
                # the attention itself on the fp16 tensor cores with the same hi/lo split (pnp_attention_fp16x3): unscaled output
                a3 = ops.attention_fp16x3(qkv.view(B, L, 3, blk.heads, hd), inv, 1.0 / math.sqrt(hd), flag, split_hi_scale=w_proj[1])
            else:
                qkv = qkv.view(B, L, 3, blk.heads, hd).permute(2, 0, 3, 1, 4)
                a = F.scaled_dot_product_attention(qkv[0], qkv[1], qkv[2], scale=inv * inv / math.sqrt(hd))
                a3 = f.split(a.transpose(1, 2).reshape(B, L, D).contiguous(), inv, w_proj, flag)
            r = f.mm(a3, w_proj)
            h = f.mm(f.ln(x, blk.norm2, w_fc1, flag, r, blk.proj.bias)[0], w_fc1)
            r, rb = f.mm(f.gelu(h, blk.fc1.bias, w_fc2, flag), w_fc2), blk.fc2.bias
        return f.ln(x, ve.norm, w["kv"], flag, r, rb, split=True, plain=want_plain)

    def _cross_kv3(self, enc3, mode="3xtf32"):
        """key(enc) / value(enc) of every cross-attention block (MED:201-221) in one GEMM -> list of (k, v, s) with k, v
        [B,L,hidden] carrying the factor s (2^11 in the fp16 form: the cross-attention takes it back, see CrossAttentionSelf)."""
        f, kv = _FORMS[mode], self._weights3(mode)["kv"]
        n = len(self.layer)
        # One persistent output buffer per shape: the text-pass CUDA graph reads K/V at fixed addresses, so the GEMM writes there
        # directly and nothing is copied.  (Passes on one stream are ordered; a pass never outlives the next one's GEMM.)
        bufs = self._cache("kv")
        M, N = enc3.shape[0] * enc3.shape[1], kv[0].shape[0]
        key = (M, N, str(enc3.device))
        if key not in bufs:
            bufs[key] = torch.empty((M, N), dtype=torch.float32, device=enc3.device)
        out = f.mm(enc3, kv, out=bufs[key]).view(enc3.shape[0], enc3.shape[1], n, 2, -1)
        return [(out[:, :, i, 0], out[:, :, i, 1], f.scale) for i in range(n)]

    def _graphed(self, key, what, inputs, run):
        """run(*inputs) replayed from the CUDA graph kept under `key`, captured on first use after two warm-ups on a side stream
        (autograd buffers, cuBLAS workspaces); `inputs` are copied into the graph's own copies of them.  -> run's result, which
        the next replay overwrites, or None when capture failed (a warning, once per key; eager is always correct)."""
        graphs = self._cache("graphs")
        if key not in graphs:
            static = [t.clone() for t in inputs]
            try:
                cur = torch.cuda.current_stream()
                side = torch.cuda.Stream()
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    for _ in range(2):
                        run(*static)
                cur.wait_stream(side)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    out = run(*static)
                graphs[key] = (g, static, out)
            except Exception as e:  # noqa: BLE001 -- a failed capture must not take the pass down
                import warnings
                warnings.warn("%s CUDA graph capture failed (%s); running it eagerly" % (what, str(e).partition("\n")[0][:200]))
                torch.cuda.synchronize()
                graphs[key] = None
        if graphs[key] is None:
            return None
        g, static, out = graphs[key]
        for s, t in zip(static, inputs):
            s.copy_(t)
        g.replay()
        return out

    USE_VIT_GRAPH = True

    def _encode(self, imgs):
        """(enc or None, per-block cross-attention (k, v, s) or [None]*n) for the current gemm_precision.  enc is None on the
        split path: a split mode, CUDA input and frozen weights."""
        mode = self.gemm_precision
        if mode in self.SPLIT_MODES and imgs.is_cuda and self._refresh():
            with torch.no_grad():
                kvs = self._encode_graphed(imgs, mode) if self.USE_VIT_GRAPH else None
                if kvs is None:
                    kvs = self._cross_kv3(self._vit3(imgs, mode=mode)[0], mode)
                return None, kvs
        return self._vit(imgs), [None] * len(self.layer)

    def _encode_graphed(self, imgs, mode):
        """The encoder pass + the K/V GEMM replayed from a CUDA graph (one per image shape): ~330 launches whose host-side issue
        otherwise leaves the GPU idle for ~3 ms per pass.  The graph's only output is the persistent K/V buffer of _cross_kv3.
        Returns None when capture is impossible here."""
        return self._graphed(("encoder", tuple(imgs.shape), str(imgs.device), mode), "encoder", (imgs,),
                             lambda x: self._cross_kv3(self._vit3(x, mode=mode)[0], mode))

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
        lin = _plain_linear if enc is not None else self._linear3
        x = self._embed(ids)
        for lyr, kv in zip(self.layer, kvs):
            x = lyr.cross_and_ffn(lyr.self_attention(x, add_mask, lin), enc, kv, lin)
        return self.itm_head(x[:, 0])

    def _text_pass(self, ids, add_mask, token_mask, enc, kvs, layer, head):
        """The text side of the trimmed GradCAM pass: BERT layers below `layer` without grad, the block's attention
        probabilities as the leaf, the loss differentiated w.r.t. them, the fused GradCAM kernel.  -> (cam [B,T-1,K-1], logits)."""
        lin = _plain_linear if enc is not None else self._linear3
        cap = GradcamCapture(head, token_mask)
        xattn = self.layer[layer].crossattention.self
        xattn.save_attention, xattn.capture, xattn.detach_probs = True, cap, True
        try:
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
        finally:
            xattn.save_attention, xattn.capture, xattn.detach_probs = False, None, False
        cap.dprobs = dprobs
        _, cam = ops.softmax_bwd_gradcam(cap.probs.detach(), dprobs.contiguous(), token_mask, head,
                                         1.0 / math.sqrt(64), need_dscores=False, need_gradcam=True)
        return cam, out.detach()

    # ---- the text pass as a CUDA graph -----------------------------------------------------------------
    USE_TEXT_GRAPH = True

    def _text_pass_graphed(self, ids, add_mask, token_mask, kvs, layer, head):
        """_text_pass replayed from a CUDA graph: the text side is ~700 launches of kernels that each run for microseconds
        (B*T = 875 rows at cfg1), so issued one by one it is bound by launch latency, not by the GPU.  One graph per
        (shapes, block, head); the K/V views of _cross_kv3's persistent buffer are read in place, the result is copied out.
        Returns None when capture is impossible here (the caller then runs the eager pass)."""
        k0, _, s0 = kvs[0]
        key = ("text", tuple(ids.shape), tuple(k0.shape), k0.data_ptr(), int(layer), int(head), float(s0), str(ids.device),
               token_mask.shape[1], self.gemm_precision)
        res = self._graphed(key, "text-pass", (ids, add_mask, token_mask), lambda *st: self._text_pass(*st, None, kvs, layer, head))
        return None if res is None else (res[0].clone(), res[1].clone())

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
        add_mask = ((1.0 - att.float()) * -10000.0)[:, None, None, :]
        if full_backward:
            cap = GradcamCapture(head, token_mask)
            xattn = self.layer[layer].crossattention.self
            xattn.save_attention, xattn.capture = True, cap
            try:
                with torch.enable_grad():
                    enc = self._vit(visual_input)
                    x = self._embed(ids)
                    for lyr in self.layer:
                        x = lyr.cross_and_ffn(lyr.self_attention(x, add_mask), enc)
                    out = self.itm_head(x[:, 0])
                    loss = out[:, 1].sum()       # BITM:399
                    self.zero_grad()
                    loss.backward()              # BITM:404; FusedXattnSoftmax.backward fills cap.gradcam
            finally:
                xattn.save_attention, xattn.capture = False, None
            cam = cap.gradcam
        else:
            with torch.no_grad():
                enc, kvs = self._encode(visual_input)
            res = self._text_pass_graphed(ids, add_mask, token_mask, kvs, layer, head) if self.USE_TEXT_GRAPH and enc is None else None
            cam, out = res if res is not None else self._text_pass(ids, add_mask, token_mask, enc, kvs, layer, head)
        P = self.patch_num
        return cam.view(B, T - 1, P, P), out.detach()
