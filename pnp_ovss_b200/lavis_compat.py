"""Bridges to the reference's LAVIS objects: checkpoints and live `BlipITM` models.

Three things a user of the reference needs when switching:

  * `load_lavis_state_dict(model, sd)` -- load the weights of the reference's LAVIS `BlipITM`
    (`model_large_retrieval_flickr.pth`, YAML:10; key layout of VIT:205-258, MED:56-82, MED:312-445, BITM:43-57) into
    `pnp_ovss_b200.blip_itm.BlipITM`, resizing the ViT position embedding the way `BaseModel.load_checkpoint` does
    (BASE:44-73, BASE:108: bicubic on the patch grid, class token kept).  `export_lavis_state_dict` is the inverse.
  * `gradcam_from_lavis_model(...)` -- GradCAM of one (block, head) from a *live* LAVIS-protocol model, i.e. one whose
    cross-attention modules sit at `model.text_encoder.base_model.base_model.encoder.layer[i].crossattention.self` and
    expose `save_attention / get_attention_map() / get_attn_gradients()` (BITM:388-425, MED:162-177).  The captured
    tensors stay on the device and go through `pnp_xattn_softmax_bwd_gradcam`; nothing is copied to the host.
  * `fused_cross_attention(model, block, head, token_mask)` -- context manager that swaps the forward of that block's
    LAVIS `BertSelfAttention` instance for one that computes MED:228-300 with the fused softmax kernel
    (`FusedXattnSoftmax`), so stage (a) runs inside an unmodified LAVIS install.

Nothing here imports LAVIS; the functions only rely on the attribute protocol quoted above."""
import contextlib
import math

import torch
import torch.nn.functional as F

from . import ops
from .blip_itm import FusedXattnSoftmax, GradcamCapture

# keys of the reference checkpoint that the ITM path never reads (ITC projections, momentum copies, queues, buffers)
_IGNORED_PREFIXES = ("vision_proj.", "text_proj.", "temp", "visual_encoder_m.", "text_encoder_m.", "vision_proj_m.",
                     "text_proj_m.", "image_queue", "text_queue", "idx_queue", "queue_ptr", "ptr_queue")
_IGNORED_SUFFIXES = ("position_ids",)


def _pairs(prefix_native, prefix_lavis, names=("weight", "bias")):
    return [("%s.%s" % (prefix_native, n), "%s.%s" % (prefix_lavis, n)) for n in names]


def native_to_lavis_keys(model):
    """{native parameter name: LAVIS checkpoint key} for a blip_itm.BlipITM."""
    m = {"visual_encoder.cls_token": "visual_encoder.cls_token", "visual_encoder.pos_embed": "visual_encoder.pos_embed",
         "word_emb.weight": "text_encoder.embeddings.word_embeddings.weight",
         "pos_emb.weight": "text_encoder.embeddings.position_embeddings.weight"}
    add = lambda a, b: m.update(_pairs(a, b))
    add("visual_encoder.patch_embed", "visual_encoder.patch_embed.proj")        # timm PatchEmbed, VIT:220
    add("visual_encoder.norm", "visual_encoder.norm")
    for i in range(len(model.visual_encoder.blocks)):                            # VIT:120-160
        n, l = "visual_encoder.blocks.%d" % i, "visual_encoder.blocks.%d" % i
        add(n + ".norm1", l + ".norm1")
        add(n + ".qkv", l + ".attn.qkv")
        add(n + ".proj", l + ".attn.proj")
        add(n + ".norm2", l + ".norm2")
        add(n + ".fc1", l + ".mlp.fc1")
        add(n + ".fc2", l + ".mlp.fc2")
    add("emb_ln", "text_encoder.embeddings.LayerNorm")                           # MED:75
    for i in range(len(model.layer)):                                            # MED:412-445
        n, l = "layer.%d" % i, "text_encoder.encoder.layer.%d" % i
        add(n + ".q", l + ".attention.self.query")
        add(n + ".k", l + ".attention.self.key")
        add(n + ".v", l + ".attention.self.value")
        add(n + ".attn_out", l + ".attention.output.dense")
        add(n + ".attn_ln", l + ".attention.output.LayerNorm")
        for p in ("query", "key", "value"):
            add(n + ".crossattention.self." + p, l + ".crossattention.self." + p)
        add(n + ".cross_out", l + ".crossattention.output.dense")
        add(n + ".cross_ln", l + ".crossattention.output.LayerNorm")
        add(n + ".inter", l + ".intermediate.dense")
        add(n + ".out", l + ".output.dense")
        add(n + ".out_ln", l + ".output.LayerNorm")
    add("itm_head", "itm_head")                                                  # BITM:57
    return m


def resize_pos_embed(pos_embed, n_tokens):
    """Position embedding [1, 1+g*g, D] of a checkpoint -> [1, n_tokens, D] (BASE:44-73): the class-token row is kept,
    the g x g grid is resampled bicubically (align_corners=False) to the model's grid."""
    if pos_embed.shape[1] == n_tokens:
        return pos_embed
    D = pos_embed.shape[-1]
    g_old = int(round(math.sqrt(pos_embed.shape[1] - 1)))
    g_new = int(round(math.sqrt(n_tokens - 1)))
    if g_old * g_old + 1 != pos_embed.shape[1] or g_new * g_new + 1 != n_tokens:
        raise ValueError("position embeddings must be 1 + square grids, got %d -> %d" % (pos_embed.shape[1], n_tokens))
    grid = pos_embed[:, 1:].reshape(1, g_old, g_old, D).permute(0, 3, 1, 2)
    grid = F.interpolate(grid.float(), size=(g_new, g_new), mode="bicubic", align_corners=False)
    return torch.cat([pos_embed[:, :1], grid.permute(0, 2, 3, 1).reshape(1, g_new * g_new, D).to(pos_embed.dtype)], 1)


def load_lavis_state_dict(model, state_dict):
    """Copy a LAVIS BlipITM checkpoint (the dict itself or {"model": dict}, BASE:103-106) into `model`.

    Every native parameter must be found with the right shape (position embedding aside, which is resized).  Extra keys
    never raise, like the reference's `load_state_dict(..., strict=False)` (BASE:112): keys the ITM path is known not to use
    (ITC projections, momentum copies, queues) are ignored silently, any other extra key is ignored with a warning.
    Returns the list of all ignored keys."""
    sd = state_dict["model"] if "model" in state_dict and isinstance(state_dict["model"], dict) else state_dict
    kmap = native_to_lavis_keys(model)
    own = model.state_dict()
    missing = [lk for lk in kmap.values() if lk not in sd]
    if missing:
        raise KeyError("checkpoint lacks %d keys of the ITM path, first: %s" % (len(missing), missing[:4]))
    known = set(kmap.values())
    ignored, unknown = [], []
    for k in sd:
        if k in known:
            continue
        (ignored if k.startswith(_IGNORED_PREFIXES) or k.endswith(_IGNORED_SUFFIXES) else unknown).append(k)
    if unknown:
        import warnings
        warnings.warn("checkpoint has %d keys this model does not use (ignored like strict=False), first: %s" % (len(unknown), unknown[:4]))
        ignored += unknown
    new = {}
    for nk, lk in kmap.items():
        t = sd[lk]
        if nk == "visual_encoder.pos_embed":
            t = resize_pos_embed(t, own[nk].shape[1])
        if tuple(t.shape) != tuple(own[nk].shape):
            raise ValueError("%s: checkpoint shape %s, model shape %s" % (lk, tuple(t.shape), tuple(own[nk].shape)))
        new[nk] = t
    model.load_state_dict(new, strict=True)
    return ignored


def export_lavis_state_dict(model):
    """state_dict of a blip_itm.BlipITM under the LAVIS key names (what load_lavis_state_dict reads)."""
    own = model.state_dict()
    return {lk: own[nk].detach().clone() for nk, lk in native_to_lavis_keys(model).items()}


# ------------------------------------------------------------------------------------------------- live LAVIS-protocol models
def cross_attention_modules(model):
    """The 12 cross-attention `self` modules, for a native BlipITM or a LAVIS-protocol model (BITM:388-392)."""
    if hasattr(model, "layer"):
        layers = model.layer
    else:
        layers = model.text_encoder.base_model.base_model.encoder.layer
    return [lyr.crossattention.self for lyr in layers]


def _fused_forward(xa, capture):
    """MED:191-311 for the cross-attention branch with absolute positions, softmax + capture fused (kernel a)."""
    orig = xa.forward

    def forward(hidden_states, attention_mask=None, head_mask=None, encoder_hidden_states=None,
                encoder_attention_mask=None, past_key_value=None, output_attentions=False):
        key_mask = None
        ok = encoder_hidden_states is not None and xa.save_attention and hidden_states.is_cuda and \
            getattr(xa, "position_embedding_type", "absolute") == "absolute"
        if ok and encoder_attention_mask is not None:
            m = encoder_attention_mask                 # the extended additive mask [B,1,1,K] of BertModel.forward
            ok = m.dim() == 4 and m.shape[1] == 1 and m.shape[2] == 1
            if ok:
                key_mask = m[:, 0, 0, :].float().contiguous()
        if not ok:
            return orig(hidden_states, attention_mask, head_mask, encoder_hidden_states, encoder_attention_mask,
                        past_key_value, output_attentions)
        q = xa.transpose_for_scores(xa.query(hidden_states))
        k = xa.transpose_for_scores(xa.key(encoder_hidden_states))
        v = xa.transpose_for_scores(xa.value(encoder_hidden_states))
        scores = torch.matmul(q, k.transpose(-1, -2))                                           # MED:228
        probs = FusedXattnSoftmax.apply(scores.float(), key_mask, 1.0 / math.sqrt(q.shape[-1]), capture)  # MED:267-274
        xa.save_attention_map(probs)                                                            # MED:281
        probs.register_hook(xa.save_attn_gradients)                                             # MED:283
        dropped = xa.dropout(probs if probs.dtype == v.dtype else probs.to(v.dtype))   # fp16/bf16 models: kernel (a) is fp32
        if head_mask is not None:
            dropped = dropped * head_mask
        ctx = torch.matmul(dropped, v).permute(0, 2, 1, 3).contiguous()                         # MED:300-304
        ctx = ctx.view(ctx.shape[0], ctx.shape[1], -1)
        return ((ctx, probs) if output_attentions else (ctx,)) + ((k, v),)

    return forward


@contextlib.contextmanager
def fused_cross_attention(model, block, head, token_mask):
    """Inside the context, block `block`'s cross-attention of a LAVIS-protocol model runs the fused softmax and fills
    the yielded GradcamCapture (probs, dprobs, gradcam [B,T-1,K-1]) during forward/backward."""
    xa = cross_attention_modules(model)[block]
    cap = GradcamCapture(head, token_mask)
    had = "forward" in xa.__dict__
    prev, prev_save = xa.__dict__.get("forward"), xa.save_attention
    xa.forward = _fused_forward(xa, cap)
    xa.save_attention = True
    try:
        yield cap
    finally:
        xa.save_attention = prev_save
        if had:
            xa.forward = prev
        else:
            del xa.forward


def _token_mask(tokenized_text, dev):
    m = tokenized_text.attention_mask
    if not isinstance(m, torch.Tensor):
        m = torch.as_tensor(m)
    return m.to(dev).long().contiguous()


def gradcam_from_lavis_model(model, visual_input, text_input, tokenized_text, layer, head, patch_num, fused=True):
    """(gradcam [B,T-1,P,P], itm_logits [B,2]) from a live LAVIS-protocol model: BITM:386-433 for the one
    (block, head) the drivers read, on the device.

    fused=True swaps that block's softmax for kernel (a) for the duration of the call; fused=False leaves the model
    untouched (its own softmax and hooks capture probs / dprobs) and only the GradCAM product runs in
    pnp_xattn_softmax_bwd_gradcam."""
    dev = visual_input.device
    token_mask = _token_mask(tokenized_text, dev)
    samples = {"image": visual_input, "text_input": text_input}

    def run():
        with torch.enable_grad():
            out = model(samples, match_head="itm")      # BITM:395
            loss = out[:, 1].sum()                       # BITM:399
            model.zero_grad()
            loss.backward()                              # BITM:404
        return out.detach()

    xa = cross_attention_modules(model)[layer]
    if fused:
        with fused_cross_attention(model, layer, head, token_mask) as cap:
            out = run()
        cam = cap.gradcam
        xa.attention_map = xa.attn_gradients = None
    else:
        prev = xa.save_attention
        xa.save_attention = True
        try:
            out = run()
        finally:
            xa.save_attention = prev
        probs, dprobs = xa.get_attention_map(), xa.get_attn_gradients()
        _, cam = ops.softmax_bwd_gradcam(probs.detach().float().contiguous(), dprobs.float().contiguous(), token_mask,
                                         int(head), 1.0 / math.sqrt(64), need_dscores=False, need_gradcam=True)
        xa.attention_map = xa.attn_gradients = None
    B, Tm1 = cam.shape[:2]
    return cam.view(B, Tm1, patch_num, patch_num), out
